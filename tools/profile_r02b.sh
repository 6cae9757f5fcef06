#!/bin/bash
# Second-half-of-round-2 profiling on one B200 (run under gpurun from the repo root): the MSM side.
#  * per-kernel launch list of an MSM at 2^20 and 2^24 (precomputed SRS), gpu__time_duration only;
#  * ncu --set full of the accumulation kernel walking tasks in length order (2^22), of the msm_binary select-sum kernel
#    and of the scatter;
#  * the bench's own launch list (same command as profiles/r02_launches_bench_ncu.*).
# CSVs -> gpurun_out/ (summaries are written under profiles/ on the authoring box with tools/ncu_summary.py).
mkdir -p gpurun_out
timeout 200 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:"msm_|precompute" -c 300 --csv \
    --log-file gpurun_out/r02b_msm_launches.csv python tools/msm_bench.py 20 24 --pre > gpurun_out/r02b_msm_launches.log 2>&1
cat > /tmp/r02b_kernels.py <<'PY'
import os, sys, numpy as np
sys.path.insert(0, "."); sys.path.insert(0, "tests")
import jolt_b200
from jolt_b200 import G1Bases, Polynomial
from oracle import bn254 as O
from oracle.coracle import rand_limbs
G = np.array(O.to_mont_limbs(1, O.Q_MOD) + O.to_mont_limbs(2, O.Q_MOD), dtype=np.uint64)
sess = jolt_b200.Session(0)
what = sys.argv[1]
n = 1 << 22
bases = G1Bases.generate_multiples(sess, G, n)
if what == "binary":
    bits = np.random.default_rng(1).integers(0, 2, size=n).astype(np.uint8)
    bases.msm_small(bits); bases.msm_small(bits)
else:
    bases.precompute()
    tab = Polynomial.new(sess, rand_limbs(3, n))
    bases.msm(tab); bases.msm(tab)
sess.synchronize()
PY
for k in acc:msm_accumulate_kernel:1 scatter:msm_scatter_kernel:1 binary:msm_select_sum_kernel:1; do
    IFS=: read what kern skip <<< "$k"   # skip: launches of the first (warm-up) MSM
    timeout 240 ncu --set full --clock-control none --import-source on -k regex:$kern -s $skip -c 1 \
        -o /tmp/r02b_$what python /tmp/r02b_kernels.py $what > gpurun_out/r02b_ncu_$what.log 2>&1
    ncu -i /tmp/r02b_$what.ncu-rep --page raw --csv > gpurun_out/r02b_${what}_raw.csv 2>/dev/null
done
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -c 800 --csv --log-file gpurun_out/r02b_launches.csv \
    python bench.py --steps 2 --warmup 1 --no-cpu-baseline --no-msm --no-kernels > gpurun_out/r02b_ncu_list.log 2>&1
ls -la gpurun_out/r02b_*
