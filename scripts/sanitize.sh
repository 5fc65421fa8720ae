#!/bin/bash
# compute-sanitizer passes over the tensor-core conv kernel (run on a machine with a B200: bash scripts/sanitize.sh):
# the production library under memcheck / synccheck / racecheck on the grouped-launch operator test and a full forward
# of the big model through the tensor-core path.
# Logs: gpurun_out/sanitize/*.log (summaries are copied to profiles/ by hand).
set -u
cd "$(dirname "$0")/.."
OUT=gpurun_out/sanitize
mkdir -p $OUT
T1="tests/test_gpu_umma.py::test_grouped_launch_equals_single_launches"
T2="tests/test_gpu_umma.py::test_score_model_forward_tensor_core"
TMO=${SAN_TIMEOUT:-420}
run() {  # name, env-prefix..., -- command
  local name=$1; shift
  echo "=== $name" | tee -a $OUT/summary.txt
  ( time timeout $TMO "$@" ) > $OUT/$name.out 2>&1
  echo "rc=$? $(tail -n 3 $OUT/$name.out | tr '\n' ' ')" | tee -a $OUT/summary.txt
}
: > $OUT/summary.txt
for tool in memcheck synccheck racecheck; do
  run ${tool}_token1_grouped compute-sanitizer --tool $tool --print-limit 20 --log-file $OUT/${tool}_token1_grouped.log python -m pytest -x -q "$T1"
done
run synccheck_token1_forward compute-sanitizer --tool synccheck --print-limit 20 --log-file $OUT/synccheck_token1_forward.log python -m pytest -x -q "$T2"
for f in $OUT/*.log; do echo "--- $f"; grep -E "ERROR SUMMARY|RACECHECK SUMMARY|Error|hazard" "$f" | sort | uniq -c | head -20; done | tee -a $OUT/summary.txt
