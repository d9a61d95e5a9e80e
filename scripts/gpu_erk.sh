#!/bin/bash
# Explicit Runge-Kutta kernel (RK23, DOP853): its GPU parity tests, scripts/profile_explicit.py (throughput, HBM share,
# single-column latency, RK23 sweep to T*), then the whole GPU suite, smoke() and a short bench line.
set -u
OUT=${1:?usage: gpu_erk.sh OUTPUT_DIR [all|short]}
mkdir -p $OUT
nvidia-smi --query-gpu=index,name,power.limit,clocks.max.sm --format=csv > $OUT/nvidia_smi.csv 2>&1
python -c "import __graft_entry__ as g; g.build()" > $OUT/build.log 2>&1; tail -1 $OUT/build.log
PT="python -m pytest -q -m gpu -p no:cacheprovider --timeout=600 --timeout-method=thread"
( time timeout 900 $PT tests/test_gpu_explicit.py ) > $OUT/pytest_explicit.log 2>&1
echo "pytest exit $?" >> $OUT/pytest_explicit.log; tail -4 $OUT/pytest_explicit.log
( time timeout 900 python scripts/profile_explicit.py 400 3 420 ) > $OUT/profile_explicit.json 2> $OUT/profile_explicit.err
echo "profile exit $?" >> $OUT/profile_explicit.err; tail -3 $OUT/profile_explicit.err
if [ "${2:-all}" = "all" ]; then
  ( time timeout 1200 $PT tests --deselect tests/test_gpu_explicit.py ) > $OUT/pytest_gpu.log 2>&1
  echo "pytest exit $?" >> $OUT/pytest_gpu.log; tail -4 $OUT/pytest_gpu.log
  timeout 200 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.log 2>&1; tail -1 $OUT/smoke.log
  ( time timeout 600 python bench.py --gpus 1 --steps 3 --warmup 1 --no-cpu-baseline --no-tstar --no-large-n ) > $OUT/bench.json 2> $OUT/bench.err
  echo "bench exit $?" >> $OUT/bench.err; tail -3 $OUT/bench.err; tail -c 600 $OUT/bench.json
fi
echo done
