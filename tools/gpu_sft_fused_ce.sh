#!/bin/bash
# The cross-entropy-from-hidden-states checks on one B200, in two parts (each takes a few minutes):
#   tools/gpu_sft_fused_ce.sh tests OUTDIR  -- the fused-CE GPU tests, the rest of the GPU suite, smoke(), tools/sft_fused_lm_head.py
#   tools/gpu_sft_fused_ce.sh extra OUTDIR  -- the fused-CE GPU tests again, bench.py, compute-sanitizer memcheck / racecheck on
#                                             the aa_ce_rows tests
# Logs and JSON results are written to OUTDIR.
set -u
if [ $# -ne 2 ]; then echo "usage: $0 tests|extra OUTDIR" >&2; exit 2; fi
OUT=$2
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/gpu_$1.txt 2>&1
cat $OUT/gpu_$1.txt
if [ "$1" = tests ]; then
  timeout 240 python -m pytest tests/test_gpu_fused_ce.py -m gpu -q -rf > $OUT/pytest_fused_ce.log 2>&1; echo "fused tests exit $?"
  tail -25 $OUT/pytest_fused_ce.log
  timeout 240 python -m pytest tests -m gpu -q -rf --ignore=tests/test_gpu_fused_ce.py > $OUT/pytest_gpu_rest.log 2>&1; echo "rest gpu exit $?"
  tail -6 $OUT/pytest_gpu_rest.log
  timeout 90 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.log 2>&1; echo "smoke exit $?"; tail -2 $OUT/smoke.log
  timeout 200 python tools/sft_fused_lm_head.py > $OUT/sft_fused_lm_head.json 2> $OUT/sft_tool.err; echo "tool exit $?"
  head -c 4000 $OUT/sft_fused_lm_head.json; tail -5 $OUT/sft_tool.err
else
  timeout 100 python -m pytest tests/test_gpu_fused_ce.py -m gpu -q -rf > $OUT/pytest_fused_ce.log 2>&1; echo "fused tests exit $?"
  tail -25 $OUT/pytest_fused_ce.log
  timeout 300 python bench.py --gpus 1 --steps 3 --warmup 1 > $OUT/bench.json 2> $OUT/bench.err; echo "bench exit $?"
  head -c 800 $OUT/bench.json; tail -3 $OUT/bench.err
  CS=$(command -v compute-sanitizer || echo /usr/local/cuda/bin/compute-sanitizer)
  if [ -x "$CS" ]; then
    for tool in memcheck racecheck; do
      timeout 100 $CS --tool $tool --error-exitcode 77 --print-limit 20 python -m pytest tests/test_gpu_fused_ce.py -m gpu -q \
        -k "compaction or out_of_range" > $OUT/sanitizer_${tool}_ce_rows.log 2>&1
      echo "$tool exit: $?"; grep -E "ERROR SUMMARY|RACECHECK SUMMARY|passed|failed" $OUT/sanitizer_${tool}_ce_rows.log | tail -3
    done
  else
    echo "no compute-sanitizer on this machine"
  fi
fi
