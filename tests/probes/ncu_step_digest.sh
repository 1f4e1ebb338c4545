#!/bin/bash
# Capture one training step's big kernels with `ncu --set full` and keep only text digests of the report in OUTDIR:
# per-kernel raw metrics + per-source-line stall digests of selected kernels (the report itself is large and is deleted).
# usage, from the repository root on a machine with Nsight Compute: tests/probes/ncu_step_digest.sh OUTDIR
set -e
OUT=${1:?usage: ncu_step_digest.sh OUTDIR}
mkdir -p "$OUT"
REP=$(mktemp -d)/r2_step_kernels
ncu --set full --import-source on --clock-control none \
    -k regex:'aggregate_tc_kernel|dgi_score|bn_relu_readout|linear_tc|linear_bwd_dx|linear_wgrad|relu_bn_bwd_reduce' \
    --launch-skip 230 --launch-count 49 -f -o $REP \
    python bench.py --steps 1 --warmup 3 --no-cpu-baseline --no-e2e --no-breakdown > $OUT/r2_ncu_step.log 2>&1
python tests/probes/ncu_digest.py $REP.ncu-rep > $OUT/r2_step_kernels_digest.txt 2>&1
for k in "aggregate_tc_kernel<.*0, .*1>" "aggregate_tc_kernel<.*0, .*2>" "aggregate_tc_kernel<.*0, .*4>" "linear_bwd_dx_tc_kernel<.*1, .*1>" "linear_wgrad_tc_kernel<.*1, .*1>" "linear_tc_kernel<.*1, .*1>" "bn_relu_readout" "dgi_score_fwd" "dgi_score_bwd" "relu_bn_bwd_reduce"; do
  echo "==== $k" >> $OUT/r2_step_kernels_lines.txt
  python tests/probes/ncu_src_lines.py $REP.ncu-rep 18 --kernel-name "regex:$k" --launch-count 1 2>&1 | cut -c1-230 >> $OUT/r2_step_kernels_lines.txt || true
done
rm -rf "$(dirname "$REP")"
