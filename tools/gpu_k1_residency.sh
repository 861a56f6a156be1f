#!/bin/bash
# The K1 forward residency / lookahead checks on one B200:
#   tools/gpu_k1_residency.sh ab OUTDIR     -- tools/k1_residency_ab.py: K1 alone on the C2 tile, every candidate shape
#   tools/gpu_k1_residency.sh check OUTDIR  -- the GPU suite, smoke(), bench.py --dump-outputs for the old launch
#                                            (--variant 70) and the default, compared file by file, then bench.py
#                                            alternating old and new, three runs each
# Logs and JSON results are written to OUTDIR.
set -u
if [ $# -ne 2 ]; then echo "usage: $0 ab|check OUTDIR" >&2; exit 2; fi
OUT=$2
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/gpu_$1.txt 2>&1
cat $OUT/gpu_$1.txt
if [ "$1" = ab ]; then
  timeout 600 python tools/k1_residency_ab.py --iters 60 --rounds 3 --shapes "${SHAPES:-70,30,0,70:32}" --out $OUT/k1_residency_ab.json \
    > $OUT/k1_residency_ab.log 2>&1; echo "ab exit $?"
  grep -E "^round|Error|error" $OUT/k1_residency_ab.log | tail -20
else
  timeout 900 python -m pytest tests -m gpu -q -rf > $OUT/pytest_gpu.log 2>&1; echo "pytest gpu exit $?"
  tail -4 $OUT/pytest_gpu.log
  timeout 120 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.log 2>&1; echo "smoke exit $?"; tail -2 $OUT/smoke.log
  D=$(mktemp -d)
  timeout 400 python bench.py --gpus 1 --steps 3 --warmup 1 --variant 70 --dump-outputs $D/old > /dev/null 2> $OUT/dump_old.err
  echo "dump old exit $?"
  timeout 400 python bench.py --gpus 1 --steps 3 --warmup 1 --dump-outputs $D/new > /dev/null 2> $OUT/dump_new.err
  echo "dump new exit $?"
  python - "$D" > $OUT/dump_diff.txt <<'EOF'
import os, sys
import numpy as np
d = sys.argv[1]
names = sorted(os.listdir(os.path.join(d, 'old')))
bad = 0
for n in names:
    a, b = np.load(os.path.join(d, 'old', n)), np.load(os.path.join(d, 'new', n))
    same_layout = a.shape == b.shape and a.dtype == b.dtype
    diff = int((a.reshape(-1).view(np.uint8) != b.reshape(-1).view(np.uint8)).sum()) if same_layout else -1
    bad += diff != 0
    print(f'{n}: shape {a.shape} {a.dtype}  differing bytes {diff}')
print(f'{len(names)} files, {bad} differ')
EOF
  tail -1 $OUT/dump_diff.txt
  rm -rf "$D"
  for i in 1 2 3; do
    timeout 400 python bench.py --gpus 1 --steps 20 --warmup 3 --variant 70 > $OUT/bench_old_$i.json 2> $OUT/bench_old_$i.err
    echo "bench old $i exit $?"
    timeout 400 python bench.py --gpus 1 --steps 20 --warmup 3 > $OUT/bench_new_$i.json 2> $OUT/bench_new_$i.err
    echo "bench new $i exit $?"
  done
  python tools/k1_residency_bench_summary.py $OUT | tee $OUT/bench_summary.txt
fi
