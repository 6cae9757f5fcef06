#!/bin/bash
# Round-2 profiling on one B200 (run under gpurun from the repo root). Under ncu the library drops to one launch per
# round (a replaying profiler cannot run a kernel that waits for host commands), so the launch list and the --set full
# captures show the per-round kernels; the resident kernel's own passes are timed on the device (%globaltimer, printed by
# tools/round_probe.py). CSVs -> gpurun_out/ (summaries are written under profiles/ on the authoring box).
mkdir -p gpurun_out
python tools/round_probe.py 22 2 > gpurun_out/r02_round_probe_22.txt 2>&1
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -c 800 --csv --log-file gpurun_out/r02_launches.csv \
    python bench.py --steps 2 --warmup 1 --no-cpu-baseline --no-msm --no-kernels > gpurun_out/r02_ncu_list.log 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k regex:fused_round_kernel -c 3 -o /tmp/r02_fused \
    python bench.py --steps 1 --warmup 1 --no-cpu-baseline --no-msm --no-kernels > gpurun_out/r02_ncu_fused.log 2>&1
ncu -i /tmp/r02_fused.ncu-rep --page raw --csv > gpurun_out/r02_fused_raw.csv 2>/dev/null
cat > /tmp/r02_kernels.py <<'PY'
import sys, numpy as np
sys.path.insert(0, "."); sys.path.insert(0, "tests")
import jolt_b200
from jolt_b200 import G1Bases, Polynomial, EqPolynomial, LOW_TO_HIGH
from oracle import bn254 as O
from oracle.coracle import rand_limbs, rand_challenge
G = np.array(O.to_mont_limbs(1, O.Q_MOD) + O.to_mont_limbs(2, O.Q_MOD), dtype=np.uint64)
sess = jolt_b200.Session(0)
what = sys.argv[1]
if what == "msm":
    n = 1 << 24
    bases = G1Bases.generate_multiples(sess, G, n)
    tab = Polynomial.new(sess, rand_limbs(3, n))
    bases.msm(tab); bases.msm(tab)
elif what == "eq":
    r = np.stack([rand_challenge(9 + i) for i in range(26)])
    EqPolynomial.evals(sess, r).free(); EqPolynomial.evals(sess, r).free()
else:
    p = Polynomial.new(sess, rand_limbs(4, 1 << 24)); p.bind_with_order(rand_challenge(1), LOW_TO_HIGH)
    p = Polynomial.new(sess, rand_limbs(4, 1 << 24)); p.bind_with_order(rand_challenge(1), LOW_TO_HIGH)
sess.synchronize()
PY
for k in msm:msm_accumulate_kernel eq:eq_stream_kernel bind:bind_kernel; do
    what=${k%%:*}; kern=${k##*:}
    timeout 300 ncu --set full --clock-control none --import-source on -k regex:$kern -s 1 -c 1 -o /tmp/r02_$what \
        python /tmp/r02_kernels.py $what > gpurun_out/r02_ncu_$what.log 2>&1
    ncu -i /tmp/r02_$what.ncu-rep --page raw --csv > gpurun_out/r02_${what}_raw.csv 2>/dev/null
done
ls -la gpurun_out/r02_*
