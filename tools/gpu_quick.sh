#!/bin/bash
# Quick GPU check after a panel-kernel change: targeted parity tests, one bench line.
mkdir -p gpurun_out
timeout 400 python -m pytest tests/test_gpu_parity.py -m gpu -x -q --timeout 120 --timeout-method=thread \
  -k "panel or golden or fast or determinism or reference_sizes or ragged or lookahead" > gpurun_out/pytest_quick.log 2>&1; echo "pytest rc=$?"; tail -4 gpurun_out/pytest_quick.log
timeout 200 python bench.py --steps 10 --warmup 3 --no-cpu > gpurun_out/bench_quick.json 2> gpurun_out/bench_quick.err; echo "bench rc=$?"; cat gpurun_out/bench_quick.json; tail -2 gpurun_out/bench_quick.err
