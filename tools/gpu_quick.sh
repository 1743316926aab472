#!/bin/bash
# Quick GPU check: parity tests + one bench line (no profiler).  usage: tools/gpu_quick.sh <tag> [extra bench args]
TAG=${1:-q}; shift
OUT=gpurun_out/$TAG
mkdir -p $OUT
timeout 900 python -m pytest tests -m gpu -x -q > $OUT/pytest_gpu.log 2>&1; echo "pytest exit $?" >> $OUT/pytest_gpu.log
tail -15 $OUT/pytest_gpu.log
timeout 600 python bench.py --steps 20 --warmup 3 --no-cpu-baseline "$@" > $OUT/bench.json 2> $OUT/bench.err; echo "bench exit $?"
tail -5 $OUT/bench.err
cat $OUT/bench.json
