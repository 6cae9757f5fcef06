#!/bin/bash
# compute-sanitizer over the MSM work of the second half of round 2 (tools/sanitize.sh covers the sumcheck side):
# task binning in shared memory, region-ordered scatter, exceptional inputs (tangent, P + (-P), identity bases, crowded
# buckets), row-batched and halving-row MSMs, the msm_binary select-sum kernel, sign-magnitude kinds.
# Usage: tools/sanitize_msm.sh [OUT_DIR]   (logs -> OUT_DIR/sanitizer_msm_*.log, default $TMPDIR/sanitizer_msm)
OUT=${1:-${TMPDIR:-/tmp}/sanitizer_msm}
mkdir -p "$OUT"
SEL='exceptional_inputs or msm_rows or binary_fast_path or batch_msm or sign_magnitude or (open_matches_oracle and (3-True or 8-True or 4-True)) or msm_matches_naive or edge_scalars'
FILES="tests/test_gpu_msm.py tests/test_gpu_compact.py tests/test_gpu_hyperkzg.py"
timeout 270 compute-sanitizer --tool memcheck --leak-check no --error-exitcode 7 \
    python -m pytest $FILES -q -x -k "$SEL" --timeout 700 > "$OUT/sanitizer_msm_memcheck.log" 2>&1
echo "memcheck rc=$?" >> "$OUT/sanitizer_msm_memcheck.log"
timeout 200 compute-sanitizer --tool racecheck --error-exitcode 7 \
    python -m pytest tests/test_gpu_msm.py tests/test_gpu_compact.py -q -x -k "exceptional_inputs or (msm_rows and 2-64) or (msm_rows and 5-256) or binary_fast_path or edge_scalars" --timeout 700 > "$OUT/sanitizer_msm_racecheck.log" 2>&1
echo "racecheck rc=$?" >> "$OUT/sanitizer_msm_racecheck.log"
for f in memcheck racecheck; do tail -n 4 "$OUT/sanitizer_msm_$f.log"; done
