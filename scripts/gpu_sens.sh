#!/bin/bash
# Forward sensitivities of the BDF kernel: their GPU tests, scripts/profile_sensitivity.py (4096 lattice columns to
# t = 0.05 with P = 0, 1, 2, 4 directions), then the whole GPU suite, smoke() and a short bench line.
set -u
OUT=${1:?usage: gpu_sens.sh OUTPUT_DIR [all|short]}
mkdir -p $OUT
nvidia-smi --query-gpu=index,name,power.limit,clocks.max.sm --format=csv > $OUT/nvidia_smi.csv 2>&1
python -c "import __graft_entry__ as g; g.build()" > $OUT/build.log 2>&1; tail -1 $OUT/build.log
PT="python -m pytest -q -m gpu -p no:cacheprovider --timeout=900 --timeout-method=thread"
( time timeout 900 $PT tests/test_gpu_sensitivity.py ) > $OUT/pytest_sens.log 2>&1
echo "pytest exit $?" >> $OUT/pytest_sens.log; tail -4 $OUT/pytest_sens.log
( time timeout 900 python scripts/profile_sensitivity.py 0.05 2 ) > $OUT/profile_sensitivity.json 2> $OUT/profile_sensitivity.err
echo "profile exit $?" >> $OUT/profile_sensitivity.err; tail -6 $OUT/profile_sensitivity.err
if [ "${2:-all}" = "all" ]; then
  ( time timeout 1500 $PT tests --deselect tests/test_gpu_sensitivity.py ) > $OUT/pytest_gpu.log 2>&1
  echo "pytest exit $?" >> $OUT/pytest_gpu.log; tail -4 $OUT/pytest_gpu.log
  timeout 200 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.log 2>&1; tail -1 $OUT/smoke.log
  ( time timeout 600 python bench.py --gpus 1 --steps 3 --warmup 1 --no-tstar --no-large-n ) > $OUT/bench.json 2> $OUT/bench.err
  echo "bench exit $?" >> $OUT/bench.err; tail -3 $OUT/bench.err; tail -c 600 $OUT/bench.json
fi
echo done
