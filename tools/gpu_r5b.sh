#!/bin/bash
# Static-sphere hoist in the state kernel: tests, then A / B timelines (in-loop and flushed) and the bench.
cd "$(dirname "$0")/.."
O=gpurun_out
mkdir -p $O
timeout 900 python -m pytest tests -m gpu -x -q > $O/pytest_gpu_r5b.log 2>&1; echo "pytest rc=$?"; tail -5 $O/pytest_gpu_r5b.log
for v in "A=1" "STOMP_B200_STATES_STATIC=0"; do
  echo "== $v"
  env $v timeout 300 python tools/timeline.py c3 40 2>&1 | tail -12
  env $v timeout 300 python tools/timeline.py c3 40 flush 2>&1 | tail -12
done > $O/r5b_state_kernel_static_div.txt 2>&1
cat $O/r5b_state_kernel_static_div.txt
for v in "A=1" "STOMP_B200_STATES_STATIC=0"; do
  echo "== c5 $v"
  env $v timeout 300 python tools/timeline.py c5 20 2>&1 | tail -12
done > $O/r5b_state_kernel_static_c5.txt 2>&1
cat $O/r5b_state_kernel_static_c5.txt
timeout 600 python bench.py > $O/bench_c3_r5b.json 2> $O/bench_c3_r5b.err; echo "bench rc=$?"; cat $O/bench_c3_r5b.json
