#!/usr/bin/env python
"""bench.py - the driver's benchmark contract for the jolt_b200 hot path.

Workload (BASELINE.json configs[1]): a complete degree-2 product sumcheck over m = 2 dense
BN254-Fr tables of 2^22 entries per GPU - round 0 eval sweep, then 21 fused bind+eval passes and
the terminal bind, one challenge round trip per round (the Fiat-Shamir sync the reference has) -
run by the C++ engine behind the C ABI (jb_prove_batch).  A "step" is one such sumcheck.

metric  : BN254 Fr field-ops/s (sumcheck bind) = 3 field ops (1 mul + 1 sub + 1 add) per bound
          output element (SURVEY.md section 8d), summed over all tables and rounds, divided by the time
          of the WHOLE sumcheck (the eval sweep's muls/adds run in the same timed region but are not
          counted; `all_field_ops_per_s` reports them too).
value   : tables resident in HBM before the timed region (a fresh copy per step, so inputs exceed L2).
e2e     : the same through the reference-facing call with HOST (pinned) tables: upload + prove +
          read back inside the timed region.
--impl reference : the CPU restatement of the reference algorithm (oracle/, OpenMP over all host
          cores) on the same workload - the reference itself is Rust and cannot be built here.
N > 1   : weak scaling - each rank owns a contiguous 2^22 block of a global 2^(22+log2 N) polynomial
          (LowToHigh binding keeps pairs local), one NCCL all-reduce of the round sums per round.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
import pathlib

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
# the CPU arm's OpenMP threads must not spin at barriers when the cgroup quota is below the thread count
os.environ.setdefault("OMP_WAIT_POLICY", "passive")

METRIC = "bn254_fr_field_ops_per_s_sumcheck_bind"
UNIT = "field-ops/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log-n", type=int, default=22, help="log2 entries per table per GPU")
    ap.add_argument("--m", type=int, default=2, help="tables in the product (degree)")
    ap.add_argument("--order", default="l2h", choices=["l2h", "h2l"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-msm", action="store_true", help="skip the secondary G1 MSM measurement")
    ap.add_argument("--msm-log-n", type=int, default=20)
    ap.add_argument("--no-kernels", action="store_true", help="skip the per-kernel roofline section (bind, eq, MSM 2^20/2^24, HyperKZG, split-eq)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def bind_ops(log_n: int, m: int) -> int:
    """3 ops per bound output; a table of 2^n entries is bound n times -> 2^n - 1 outputs."""
    return 3 * m * ((1 << log_n) - 1)


def all_ops(log_n: int, m: int) -> int:
    """bind ops + eval-sweep ops: per pair index m subs, (m+1)(m-1) muls, m*m adds, m+1 accumulates."""
    total = bind_ops(log_n, m)
    per_pair = m + (m + 1) * (m - 1) + m * m + (m + 1)
    for k in range(log_n):  # round k sweeps 2^(log_n-k-1) pairs
        total += per_pair * (1 << (log_n - k - 1))
    return total


def config(args, world):
    return {
        "workload": f"product sumcheck, m={args.m} tables x 2^{args.log_n} BN254 Fr per GPU, degree {args.m}, "
                    f"all {args.log_n} rounds fused bind+eval, 125-bit challenges, order={args.order}",
        "log_n_per_gpu": args.log_n, "m": args.m, "order": args.order,
        "global_log_n": args.log_n + (world.bit_length() - 1),
        "field_ops_counted": "3 per bound output element (1 mul + 1 sub + 1 add), SURVEY 8d",
        "l2": "a fresh input copy per step; per-step inputs (m x 2^n x 32 B) exceed the 126 MB L2",
        "parallelism": f"index-sharded x{world}" if world > 1 else "single GPU",
    }


def dump_outputs(out_dir: str, res, fe) -> None:
    """--dump-outputs: what the last timed step handed its caller (jb_prove_batch's results and the member's final
    evaluations), so that two builds can be compared output for output. Every BN254 Fr value is written canonical
    (out of Montgomery form) as 8 little-endian 32-bit words in float64, which holds each word exactly:
    challenges (rounds, 8), final_claim (8,), member_claims (1, 8), round_polys (rounds, m + 1, 8; unused
    coefficient slots are 0), final_evals (m, 8)."""
    import numpy as np
    from jolt_b200 import field as F
    ch, fin, mc, rp = res
    out = pathlib.Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    total = 0
    for name, limbs in (("challenges", ch), ("final_claim", fin), ("member_claims", mc), ("round_polys", rp),
                        ("final_evals", fe)):
        limbs = np.asarray(limbs, dtype=np.uint64)
        words = [[(v >> (32 * k)) & 0xFFFFFFFF for k in range(8)] for v in F.limbs_to_ints(limbs)]
        arr = np.array(words, dtype=np.float64).reshape(limbs.shape[:-1] + (8,))
        total += arr.nbytes
        np.save(out / f"{name}.npy", arr)
    assert total <= 64 << 20, f"--dump-outputs: {total} bytes"


# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (NVML, ~2 ms period; the
    nvidia-smi loop of B200_PROFILING.md is too coarse for a timed region of tens of ms)."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.smax, self._stop = [], set(), None, False
        self.thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
        except Exception:
            self.thread = None

    def _run(self):
        nv = self.nv
        bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        while not self._stop:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def restart(self):
        """forget what was sampled so far (the timed region starts now)"""
        self.samples, self.reasons = [], set()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.smax, "reasons": [], "samples": 0}
        if self.thread is None:
            return out
        self._stop = True
        self.thread.join(timeout=2)
        if self.samples:
            s = sorted(self.samples)
            out.update(sm_mhz=s[len(s) // 2], reasons=sorted(self.reasons), samples=len(s))
        return out


# ---------------------------------------------------------------------------------------------------
def host_threads() -> int:
    """Threads the CPU arm can really use: the scheduler affinity capped by the cgroup CPU quota (the GPU
    boxes expose 128 logical CPUs under a 16-CPU quota; 128 spinning OpenMP threads on that quota are 12x
    SLOWER than 32). Twice the quota measured best (threads that block at barriers yield their share)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = int(q) / int(period)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / period
        except Exception:
            pass
    if quota:
        n = max(1, min(n, int(2 * quota + 0.5)))
    return n


def cpu_sumcheck_times(log_n: int, m: int, order: int, threads: int, reps: int) -> list[float]:
    """`reps` full sumchecks of the workload on the host cores with the C restatement of the reference
    algorithm (bind pass + eval pass per round, OpenMP static chunks of >= 1024 like Rayon's PAR_THRESHOLD).
    Returns the seconds of every repetition; the first one pays the page faults of freshly mapped buffers
    (the Rust prover's allocator is warm in steady state), so callers discard it as warm-up."""
    from oracle import coracle as C
    from oracle.coracle import rand_limbs, rand_challenge
    tabs0 = [rand_limbs(0xB200 + j, 1 << log_n) for j in range(m)]
    out = []
    for _ in range(reps):
        tabs = [t.copy() for t in tabs0]
        t0 = time.perf_counter()
        bind = None
        for rnd in range(log_n):
            if bind is not None:
                tabs = [C.bind(t, bind, order, threads) for t in tabs]
            C.product_round_evals(tabs, m, order, threads)
            bind = rand_challenge(1000 + rnd)
        tabs = [C.bind(t, bind, order, threads) for t in tabs]
        out.append(time.perf_counter() - t0)
    return out


def cpu_sumcheck_sample(log_n: int, m: int, order: int, threads: int, reps: int):
    """Best steady-state repetition (one extra warm-up repetition is run and dropped)."""
    return min(cpu_sumcheck_times(log_n, m, order, threads, reps + 1)[1:])


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port) on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    order = 1 if args.order == "l2h" else 0
    world = args.gpus
    # bounded sample: the per-GPU workload (2^log_n); warm-up and timed repetitions in ONE run so the timed
    # ones see a warm allocator (first-touch page faults of fresh 64-128 MiB buffers cost ~10x on 64 threads)
    # --steps is honoured as given (--warmup too, with at least one warm-up); one step (a full 2^log_n sumcheck)
    # takes ~0.2 s on the host cores of a B200 machine, so the default 50 + 5 ends within a minute
    total = args.steps
    nwarm = max(1, args.warmup)
    secs = cpu_sumcheck_times(args.log_n, args.m, order, threads, nwarm + total)[nwarm:]
    per = sum(secs) / len(secs)
    value = bind_ops(args.log_n, args.m) / per
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": total,
        "warmup": nwarm, "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64 (4-limb 256-bit Montgomery integers)", "data": "synthetic",
        "config": config(args, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"mean of {total} full 2^{args.log_n} m={args.m} sumchecks after {nwarm} warm-up (bind pass + eval pass per round) - "
                                   f"the per-GPU share of the workload, a bounded sample when n_gpus > 1 (field-ops/s does not depend on which "
                                   f"2^{args.log_n} block is swept); C restatement of the reference algorithm with OpenMP, not the Rust binary"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "all_field_ops_per_s": all_ops(args.log_n, args.m) / per,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
def msm_section(sess, log_n: int, with_cpu: bool):
    """Secondary metric of BASELINE.json: BN254 G1 MSM terms/s (config 3). Synthetic bases (i+1)*G generated
    on the device, uniform 253-bit scalars resident in HBM. Reported with the SRS as uploaded and with
    jb_srs_precompute; the two device results must agree, and (cpu_baseline leg) must equal the CPU port's."""
    import numpy as np
    from jolt_b200 import G1Bases, Polynomial, g1_jacobian_to_affine
    from jolt_b200 import field as F
    n = 1 << log_n
    G = np.concatenate([F.to_limbs(1, F.Q_MOD), F.to_limbs(2, F.Q_MOD)])
    rng = np.random.Generator(np.random.PCG64(0x5CA1A2))
    sc = rng.integers(0, 1 << 64, size=(n, 4), dtype=np.uint64)
    sc[:, 3] &= np.uint64(((1 << 64) - 1) >> 3)
    tab = Polynomial.new(sess, sc)
    out = {"log_n": log_n, "unit": "terms/s", "data": "synthetic: bases (i+1)*G, uniform 253-bit scalars"}
    for label, pre in (("plain_srs", False), ("precomputed_srs", True)):
        bases = G1Bases.generate_multiples(sess, G, n)
        if pre:
            bases.precompute()
        res = bases.msm(tab)
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            res = bases.msm(tab)
            ts.append(time.perf_counter() - t0)
        out[label] = {"ms": min(ts) * 1e3, "terms_per_s": n / min(ts)}
        if label == "plain_srs":
            gpu_pt = g1_jacobian_to_affine(res)
            xy = bases.affine() if with_cpu else None
            # primitive-integer columns (legacy msm_u64 / msm_u8, SURVEY 8d config 3's small-scalar variant): host
            # scalars, so the H2D of 8 / 1 bytes per term is inside the time
            small = {}
            for name, col in (("u64", sc[:, 0].copy()), ("u8", (sc[:, 1] & np.uint64(0xFF)).astype(np.uint8))):
                bases.msm_small(col)
                tt = []
                for _ in range(3):
                    t0 = time.perf_counter()
                    bases.msm_small(col)
                    tt.append(time.perf_counter() - t0)
                small[name] = {"ms": min(tt) * 1e3, "terms_per_s": n / min(tt)}
            out["small_scalars_host"] = small
        else:
            out["results_agree"] = gpu_pt == g1_jacobian_to_affine(res)
        bases.free()
    if with_cpu:
        from oracle import coracle as C
        from oracle import bn254 as O
        dts = []
        for _ in range(4):  # one warm-up (first-touch page faults, thread start-up) + best of 3
            t0 = time.perf_counter()
            cpu_xy, cpu_inf = C.g1_msm_pippenger(xy, sc, 0, host_threads())
            dts.append(time.perf_counter() - t0)
        dt = min(dts[1:])
        out["cpu_baseline"] = {"ms": dt * 1e3, "terms_per_s": n / dt, "cores": host_threads(), "kind": "port",
                               "sample": "best of 3 after 1 warm-up: Pippenger MSM (arkworks window heuristic) with the C restatement, OpenMP over windows"}
        out["matches_cpu_port"] = (not cpu_inf) and gpu_pt == (
            O.from_mont_limbs(cpu_xy[:4], O.Q_MOD), O.from_mont_limbs(cpu_xy[4:], O.Q_MOD))
    tab.free()
    return out


def kernels_section(sess, peak_hbm: float, with_cpu: bool):
    """Every streaming kernel of the path against its roofline, on ONE GPU, timed with CUDA events on the launching
    stream (best of 5 after a warm-up, a 512 MiB L2 flush between repetitions). HBM-bound kernels report algorithmic
    GB/s over the measured copy peak; the MSM bucket accumulation is integer-bound and reports bucket additions/s over
    the measured Montgomery-product ceiling (jb_diag_mul_throughput, 10 Fq products per mixed XYZZ addition)."""
    import ctypes
    import numpy as np
    import torch
    from jolt_b200 import BatchMember, EqPolynomial, EqProductMember, G1Bases, HyperKZG, LOW_TO_HIGH, HIGH_TO_LOW, Polynomial
    from jolt_b200 import field as F
    from oracle.coracle import rand_challenge, rand_limbs
    out = {"timing": "CUDA events on the launching stream, best of 5 after 1 warm-up, 512 MiB L2 flush between repetitions"}
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")

    def timed(fn, setup=None, reps=5, teardown=None):
        best = 1e30
        for rep in range(reps + 1):
            arg = setup() if setup else None
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn(arg)
            e1.record()
            e1.synchronize()
            if rep:
                best = min(best, e0.elapsed_time(e1))
            if teardown:  # hand the tables back: the next repetition's device allocations come out of the pool
                teardown(arg)
        return best

    def synth(n, seed):
        g = torch.Generator(device="cuda").manual_seed(seed)
        t = torch.randint(0, 2 ** 62, (n, 4), dtype=torch.int64, device="cuda", generator=g)
        t[:, 3] &= (1 << 60) - 1
        return t

    # the integer ceiling everything multiplier-bound is scored against
    g_mul = {}
    for name, field, variant in (("fr_full", 0, 0), ("fr_challenge125", 0, 1), ("fq_full", 1, 0)):
        v = ctypes.c_double()
        sess.check(sess.lib.jb_diag_mul_throughput(sess.h, field, variant, 2000, 148 * 8, ctypes.byref(v)))
        g_mul[name] = v.value
    out["montgomery_products_per_s"] = {k: v * 1e9 for k, v in g_mul.items()}

    # ---- bind_kernel, 2^24 (Polynomial::bind_with_order) -----------------------------------------
    n = 1 << 24
    src = synth(n, 0xB1D)
    binds = []
    for order, oname in ((LOW_TO_HIGH, "l2h"), (HIGH_TO_LOW, "h2l")):
        for ch, cname in ((rand_challenge(5), "challenge125"), (F.to_limbs(F.R_MOD - 12345), "full254")):
            def setup():
                buf = src.clone()
                return buf, Polynomial.wrap_device(sess, buf.data_ptr(), n)
            ms = timed(lambda a: a[1].bind_with_order(ch, order), setup, teardown=lambda a: a[1].free())
            gbs = 48 * n / (ms * 1e-3) / 1e9
            binds.append({"order": oname, "scalar": cname, "ms": ms, "gb_per_s": gbs, "frac_of_hbm_peak": gbs / peak_hbm})
    out["bind_kernel_2^24"] = {"algorithmic_bytes": 48 * n, "bound": "hbm", "peak": peak_hbm, "runs": binds}
    del src

    # ---- eq_stream_kernel (EqPolynomial::evals): 32 B written per output -------------------------
    eqs = []
    for lg in (22, 26):
        for cname in ("challenge125", "full254"):
            r = np.stack([rand_challenge(9 + i) if cname == "challenge125" else F.to_limbs((0x1234567 + i) * 0x9E3779B97F4A7C15 % F.R_MOD)
                          for i in range(lg)])
            ms = timed(lambda a: EqPolynomial.evals(sess, r).free())
            gbs = 32 * (1 << lg) / (ms * 1e-3) / 1e9
            ceiling = (g_mul["fr_challenge125"] if cname == "challenge125" else g_mul["fr_full"]) * 32  # GB/s if 1 product/output
            eqs.append({"log_n": lg, "point": cname, "ms": ms, "gb_per_s": gbs, "frac_of_hbm_peak": gbs / peak_hbm,
                        "integer_ceiling_gb_per_s": ceiling, "frac_of_integer_ceiling": gbs / ceiling})
    out["eq_stream_kernel"] = {"algorithmic_bytes_per_output": 32, "bound": "hbm (125-bit point) / integer pipe (254-bit point: one product per output)",
                               "peak": peak_hbm, "runs": eqs}

    # ---- G1 MSM: whole call + the bucket accumulation kernel (integer-bound) ---------------------
    G = np.concatenate([F.to_limbs(1, F.Q_MOD), F.to_limbs(2, F.Q_MOD)])
    msms = []
    for lg in (20, 24):
        nn = 1 << lg
        rng = np.random.Generator(np.random.PCG64(0x5CA1A2 + lg))
        sc = rng.integers(0, 1 << 64, size=(nn, 4), dtype=np.uint64)
        sc[:, 3] &= np.uint64(((1 << 64) - 1) >> 3)
        tab = Polynomial.new(sess, sc)
        bases = G1Bases.generate_multiples(sess, G, nn)
        # closed form (bases (i + 1) G): msm(s) == (sum_i s_i (i + 1)) G, checked on the host with one scalar multiplication
        for label in ("plain_srs", "precomputed_srs"):
            if label == "precomputed_srs":
                try:
                    bases.precompute()
                except Exception as e:  # 12 x the SRS in HBM: report, do not fail the bench
                    msms.append({"log_n": lg, "srs": label, "skipped": str(e)})
                    continue
            sess.timing_enable(True, min_items=1)
            sess.timing_collect()
            ms = timed(lambda a: bases.msm(tab), reps=3)
            acc = [t for t in sess.timing_collect() if t["kind"] == "msm_accumulate"]
            sess.timing_enable(False)
            acc_ms = min(t["ms"] for t in acc) if acc else None
            c_bits = acc[0]["m"] % 100 if acc else None
            ba_levels = acc[0]["m"] // 100 if acc else 0   # batched-affine levels in front of the XYZZ accumulation
            windows = -(-254 // c_bits) if c_bits else None
            adds = nn * windows if windows else None
            row = {"log_n": lg, "srs": label, "ms": ms, "terms_per_s": nn / (ms * 1e-3), "window_bits": c_bits, "windows": windows,
                   "accumulate_kernel_ms": acc_ms, "batched_affine_levels": ba_levels}
            if acc_ms:
                rate = adds / (acc_ms * 1e-3)
                # Fq products per bucket addition: 10 for a mixed XYZZ addition; with L affine levels the share
                # 1 - 2^-L of the additions costs ~6.3 (5M + 1S + the prefix / peel products of the shared inversion)
                per_add = 10.0 if not ba_levels else 6.3 * (1 - 0.5 ** ba_levels) + 10.0 * 0.5 ** ba_levels
                ceiling = g_mul["fq_full"] * 1e9 / per_add
                row.update(bucket_adds_per_s=rate, fq_products_per_addition=per_add, integer_ceiling_adds_per_s=ceiling,
                           frac_of_integer_ceiling=rate / ceiling,
                           hbm_gb_per_s=(adds * 68) / (acc_ms * 1e-3) / 1e9, frac_of_hbm_peak=(adds * 68) / (acc_ms * 1e-3) / 1e9 / peak_hbm)
            msms.append(row)
        bases.free()
        tab.free()
    out["msm_g1"] = {"bound": "integer pipe (10 Fq products per mixed XYZZ bucket addition, ~6.3 per batched-affine addition); 68 B gathered per addition",
                     "accumulate_kernel_ms": "batched-affine levels (if any) + the XYZZ accumulation kernel", "runs": msms}

    # ---- row-batched small-scalar MSM (Dory tier-1 rows) and a binary column ---------------------
    try:
        rows_n, row_w = 1024, 4096
        bases = G1Bases.generate_multiples(sess, G, 1 << 22)
        rngm = np.random.Generator(np.random.PCG64(0xD0))
        mat = rngm.integers(0, 1 << 64, size=rows_n * row_w, dtype=np.uint64)
        bases.msm_rows(mat, rows_n)  # builds the 8-bit window table of the first row_w bases once
        t_rows = timed(lambda a: bases.msm_rows(mat, rows_n), reps=3)
        t_loop = timed(lambda a: [bases.msm_small(mat[r * row_w:(r + 1) * row_w]) for r in range(16)], reps=2) / 16 * rows_n
        bits = rngm.integers(0, 2, size=1 << 22, dtype=np.uint8)
        bases.msm_small(bits)
        t_bin = timed(lambda a: bases.msm_small(bits), reps=3)
        out["msm_rows_u64_1024x4096"] = {"ms": t_rows, "terms_per_s": rows_n * row_w / (t_rows * 1e-3), "row_by_row_ms_extrapolated_from_16_rows": t_loop,
                                         "note": "jb_msm_g1_rows: host scalars (H2D of 8 B/term inside), one pipeline pass over (row, bucket) sets"}
        out["msm_binary_2^22"] = {"ms": t_bin, "terms_per_s": (1 << 22) / (t_bin * 1e-3), "note": "msm_binary arm: host flags (1 B/term H2D inside), select-sum kernel"}
        bases.free()
    except Exception as e:  # secondary lines: report, do not fail the bench
        out["msm_rows_u64_1024x4096"] = {"skipped": str(e)}

    # ---- HyperKZG open, ell = 22 (precomputed SRS) ----------------------------------------------
    ell = 22
    nn = 1 << ell
    bases = G1Bases.generate_multiples(sess, G, nn)
    bases.precompute()
    poly = Polynomial.new(sess, rand_limbs(1, nn))
    point = np.stack([rand_challenge(7 + i) for i in range(ell)])
    tc = timed(lambda a: HyperKZG.commit(bases, poly), reps=3)
    to = timed(lambda a: HyperKZG.open(bases, poly, point, lambda c: 12345, lambda v: 6789), reps=3)
    out["hyperkzg_ell22"] = {"commit_ms": tc, "open_ms": to, "srs": "precomputed windows + small-MSM table",
                             "bound": "integer pipe (MSMs)", "note": "ell - 1 folds, ell - 1 + 3 MSMs, 3 Horner scans, two transcript callbacks"}
    bases.free()
    poly.free()

    # ---- split-eq (Gruen) member, 2^22, m = 2 (degree 3) ----------------------------------------
    lg = 22
    nn = 1 << lg
    tabs = [synth(nn, 0xE0 + j) for j in range(2)]
    w = np.stack([rand_challenge(100 + i) for i in range(lg)])
    eqp = EqPolynomial.evals(sess, w)
    from jolt_b200 import ProductMember
    probe_bufs = [t.clone() for t in tabs]
    probe = ProductMember(sess, [eqp] + [Polynomial.wrap_device(sess, t.data_ptr(), nn) for t in probe_bufs], LOW_TO_HIGH)
    ev = probe.prove_round_evals(None, 0)
    claim = (ev[0] + ev[1]) % F.R_MOD
    probe.close()
    del probe_bufs

    def se_setup():
        bufs = [t.clone() for t in tabs]
        return bufs, EqProductMember(sess, [Polynomial.wrap_device(sess, b.data_ptr(), nn) for b in bufs], w)

    def se_run(a):
        jolt_b200.prove_batch_native([BatchMember(claim, 1, lg, 0)], [a[1]], lg, 3, claim, seed=9, raw=True)
        a[1].close()
    import jolt_b200
    ms = timed(se_run, se_setup, reps=3)
    alg = 2 * 96 * nn  # two witness tables bound over the whole sumcheck (~96 N bytes each); no eq table is streamed
    out["split_eq_member_2^22_m2"] = {"ms": ms, "algorithmic_bytes": alg, "gb_per_s": alg / (ms * 1e-3) / 1e9,
                                      "frac_of_hbm_peak": alg / (ms * 1e-3) / 1e9 / peak_hbm, "bound": "hbm nominal; latency (22 round trips) in practice"}
    del flush
    return out


def run_ours(args):
    import numpy as np
    import torch
    import jolt_b200
    from jolt_b200 import BatchMember, Polynomial, ProductMember
    from jolt_b200 import field as F

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - jolt_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sess = jolt_b200.Session(local, cuda_stream=stream.cuda_stream)
    order = jolt_b200.LOW_TO_HIGH if args.order == "l2h" else jolt_b200.HIGH_TO_LOW
    n = 1 << args.log_n
    m = args.m
    K, W = args.steps, args.warmup

    def synth(seed):
        g = torch.Generator(device="cuda").manual_seed(seed)
        t = torch.randint(0, 2 ** 62, (n, 4), dtype=torch.int64, device="cuda", generator=g)
        t[:, 3] &= (1 << 60) - 1  # raw value < 2^252 < r: canonical Montgomery limbs
        return t

    parity = None
    if world > 1:
        # each rank's synthetic tables ARE its shard: the contiguous block of the global tables under LowToHigh,
        # the strided slice under HighToLow (jb_sharded_member_create)
        from jolt_b200.dist import init_comm, parity_self_check, prove_sharded, sharded_claim
        init_comm(sess, dist)
        # before anything is timed: the sharded proof must equal the single-GPU proof of the same global polynomial
        parity = parity_self_check(sess, dist, log_n=14, m=m, order=order)
        if rank == 0 and not parity.get("identical_to_single_gpu"):
            raise SystemExit(f"bench.py: sharded proof differs from the single-GPU proof: {parity}")

    def one_step(bufs, seed):
        polys = [Polynomial.wrap_device(sess, b.data_ptr(), n) for b in bufs]
        if world == 1:
            mem = ProductMember(sess, polys, order)
            res = jolt_b200.prove_batch_native(desc, [mem], args.log_n, m, claim, seed=seed, raw=True)
            fe = mem.final_evals(raw=True)
            mem.close()
        else:
            res, fe = prove_sharded(sess, polys, claim, seed, raw=True, order=order)
        return res, fe

    # ---- value arm: inputs resident in HBM, one fresh copy per step ------------------------------
    base = [synth(0xB200 + 16 * rank + j) for j in range(m)]
    # the input claim (known from the previous protocol stage in a real proof): sum_x prod_j f_j(x)
    if world == 1:
        probe_bufs = [b.clone() for b in base]  # (kept alive: a wrapped table borrows the tensor's memory)
        probe = ProductMember(sess, [Polynomial.wrap_device(sess, b.data_ptr(), n) for b in probe_bufs], order)
        ev = probe.prove_round_evals(None, 0)
        claim = (ev[0] + ev[1]) % F.R_MOD
        probe.close()
        del probe_bufs
    else:
        claim = sharded_claim(sess, [Polynomial.wrap_device(sess, b.data_ptr(), n) for b in base], dist)
    desc = [BatchMember(claim, 1, args.log_n, 0)]
    copies = [[b.clone() for b in base] for _ in range(K + W)]
    torch.cuda.synchronize()
    # the NVML sampler thread starts BEFORE the warm-up (its initialisation takes tens of ms: started between the
    # barrier and the first event it made rank 0 late and every other rank's first exchange wait for it, inside their
    # timed region); its samples are discarded at the start of the timed region
    sampler = ClockSampler(local) if rank == 0 else None
    for w in range(W):
        one_step(copies[w], 7)
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    sess.timing_enable(True, min_items=1 << (args.log_n - 3))
    launches0 = sess.launch_count
    if sampler:
        sampler.restart()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    t0 = time.perf_counter()
    for k in range(K):
        res, fe = one_step(copies[W + k], 7)
    e1.record(stream)
    e1.synchronize()
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    dev_ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, fe)
    launches = sess.launch_count - launches0
    timed = sess.timing_collect()
    sess.timing_enable(False)
    if dist:
        tmax = torch.tensor([dev_ms], device="cuda")
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dev_ms = float(tmax.item())
    del copies

    # ---- e2e arm: host (pinned) tables -> upload -> prove -> read back ------------------------------
    host = [b.cpu().pin_memory() for b in base]
    host_np = [h.numpy().view(np.uint64) for h in host]

    def e2e_step():
        polys = [Polynomial.new(sess, h) for h in host_np]
        if world == 1:
            mem = ProductMember(sess, polys, order)
            res = jolt_b200.prove_batch_native(desc, [mem], args.log_n, m, claim, seed=7, raw=True)
            fe = mem.final_evals(raw=True)
            mem.close()
        else:
            res, fe = prove_sharded(sess, polys, claim, 7, raw=True, order=order)
        return res, fe

    e2e_res, e2e_fe = e2e_step()
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    Ke = max(3, min(K, 10))
    t0 = time.perf_counter()
    for _ in range(Ke):
        e2e_res, e2e_fe = e2e_step()
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / Ke
    if dist:
        tmax = torch.tensor([e2e_s], device="cuda")
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        e2e_s = float(tmax.item())
    # same inputs + same stand-in transcript => identical proofs through both arms
    assert all((a == b).all() for a, b in zip(e2e_res, res)) and (e2e_fe == fe).all(), "value arm and e2e arm disagree"
    # the full-size timed run must end where a sumcheck has to: final claim == prod_j f_j(point)
    fin_claim = F.from_limbs(res[1])
    prod = 1
    for v in F.limbs_to_ints(fe):
        prod = prod * v % F.R_MOD
    assert prod == fin_claim, "full-size run: final claim != product of the final evaluations"
    if parity is not None:
        parity["full_size_final_claim_is_product_of_final_evals"] = True

    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return

    ms_per_step = dev_ms / K
    ops_step = bind_ops(args.log_n, m) * world
    value = ops_step / (ms_per_step * 1e-3)
    # ---- roofline of the dominant kernel: the largest fused bind+eval pass -------------------------
    peaks = {}
    try:
        peaks = json.load(open(ROOT / "MEASURED_PEAKS.json"))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)
    big = [t for t in timed if t["kind"] == "fused_bind_eval" and t["items"] == n // 4]
    roof = None
    if big:
        avg_ms = sum(t["ms"] for t in big) / len(big)
        alg_bytes = m * 48 * n  # per table: read 2^n x 32 B, write 2^(n-1) x 32 B
        ach = alg_bytes / (avg_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": f"fused_round_kernel<M={m},{args.order},BIND,HI4> (round 1: 2^{args.log_n} -> 2^{args.log_n - 1})",
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
                "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": avg_ms, "launches_timed": len(big),
                "traffic": None}
        try:  # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed ncu --set full capture
            tr = json.load(open(ROOT / "profiles" / "r01b_traffic.json"))
            if args.log_n == 22 and m == 2 and args.order == "l2h":
                roof["traffic"] = tr["fused_round_kernel m=2 l2h 2^22"]["traffic"]
                roof["traffic_source"] = tr["source"]
        except Exception:
            pass
        kernel_ms = sum(t["ms"] for t in timed) / K
        roof["timed_kernels_share_of_step"] = kernel_ms / ms_per_step
        # every timed streaming pass of a step (CUDA events on the launching stream, averaged over the K steps):
        # algorithmic bytes = m x 64 B read per pair (eval-only) or m x 192 B per pair (bind + eval: 4 reads, 2 writes)
        groups = {}
        for t in timed:
            groups.setdefault((t["kind"], t["items"]), []).append(t["ms"])
        roof["passes"] = [
            {"kind": k, "pairs": it, "avg_ms": sum(v) / len(v),
             "gb_per_s": (m * (192 if k == "fused_bind_eval" else 64) * it) / (sum(v) / len(v) * 1e-3) / 1e9,
             "frac_of_peak": (m * (192 if k == "fused_bind_eval" else 64) * it) / (sum(v) / len(v) * 1e-3) / 1e9 / peak}
            for (k, it), v in sorted(groups.items(), key=lambda kv: -kv[0][1]) if k in ("fused_bind_eval", "eval_only")]

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32 (8-limb 256-bit Montgomery integers)", "data": "synthetic",
        "config": config(args, world),
        "e2e": {"value": ops_step / e2e_s, "unit": UNIT, "ms_per_step": e2e_s * 1e3,
                "h2d_bytes_per_step": m * n * 32 * world,
                "d2h_bytes_per_step": (args.log_n * (m + 1) * 32 + m * 32) * world},
        "gpu_launches": int(launches),
        "parity_checked": parity if parity is not None else {
            "full_size_final_claim_is_product_of_final_evals": True, "value_arm_equals_e2e_arm": True,
            "note": "N = 1: bit-exact parity against the oracle is tests/ (-m gpu); the bench asserts the sumcheck identity"},
        "clocks": clocks,
        "roofline": roof,
        "all_field_ops_per_s": all_ops(args.log_n, m) * world / (ms_per_step * 1e-3),
        "wall_ms_per_step": wall / K * 1e3,
    }
    if world == 1:
        # Secondary, NOT the headline: the same sumcheck when the tables arrive as compact u64 columns
        # (Polynomial<u64>, what most witness columns are) and are promoted on the device: 8 B/entry over PCIe
        # instead of 32. Cross-checked against the field-element path on the promoted values.
        g = torch.Generator().manual_seed(0xC0)
        cols = [torch.randint(-(2 ** 63), 2 ** 63 - 1, (n,), dtype=torch.int64, generator=g).pin_memory() for _ in range(m)]
        cols_np = [c.numpy().view(np.uint64) for c in cols]

        def compact_step(promoted=None):
            polys = [Polynomial.new(sess, q) for q in promoted] if promoted else [Polynomial.from_small(sess, c) for c in cols_np]
            mem = ProductMember(sess, polys, order)
            r = jolt_b200.prove_batch_native(cdesc, [mem], args.log_n, m, cclaim, seed=7, raw=True)
            f = mem.final_evals(raw=True)
            mem.close()
            return r, f

        probe = ProductMember(sess, [Polynomial.from_small(sess, c) for c in cols_np], order)
        ev = probe.prove_round_evals(None, 0)
        cclaim = (ev[0] + ev[1]) % F.R_MOD
        probe.close()
        cdesc = [BatchMember(cclaim, 1, args.log_n, 0)]
        promoted = []
        for c in cols_np:
            q = Polynomial.from_small(sess, c)
            promoted.append(q.evals())
            q.free()
        ref_r, ref_f = compact_step(promoted)
        cr, cf = compact_step()
        agree = all((a == b).all() for a, b in zip(cr, ref_r)) and (cf == ref_f).all()
        del promoted
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(5):
            compact_step()
        torch.cuda.synchronize()
        cs = (time.perf_counter() - t0) / 5
        line["e2e_compact_u64"] = {"value": ops_step / cs, "unit": UNIT, "ms_per_step": cs * 1e3,
                                   "h2d_bytes_per_step": m * n * 8, "matches_field_path": bool(agree),
                                   "note": "secondary: u64 columns promoted on the device (jb_table_upload_small), not the headline workload"}
    if world == 1 and not args.no_msm:
        line["msm"] = msm_section(sess, args.msm_log_n, not args.no_cpu_baseline)
    if world == 1 and not args.no_kernels:
        line["kernels"] = kernels_section(sess, peak, not args.no_cpu_baseline)
    if world == 1 and not args.no_cpu_baseline:
        threads = host_threads()
        reps = 2
        secs = cpu_sumcheck_sample(args.log_n, m, 1 if args.order == "l2h" else 0, threads, reps)
        line["cpu_baseline"] = {
            "value": bind_ops(args.log_n, m) / secs, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"best of {reps} (after 1 warm-up) full 2^{args.log_n} m={m} sumchecks with the C restatement of the reference "
                      "algorithm (oracle/oracle.c, OpenMP); the Rust reference cannot be built in this image"}
    print(json.dumps(line), flush=True)
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
