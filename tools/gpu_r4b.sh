#!/bin/bash
# visit r4b: paced solve loop + pair rule inside the specialised kernel
cd "$(dirname "$0")/.."
O=gpurun_out
python -m pytest tests/test_self_collision.py tests/test_gpu_parity.py -m gpu -x -q > $O/pytest_gpu_r4b.log 2>&1; tail -5 $O/pytest_gpu_r4b.log
python tools/e2e_breakdown.py c3 60 20 8 > $O/e2e_breakdown_r4b.txt 2>&1; cat $O/e2e_breakdown_r4b.txt
STOMP_B200_SOLVE_AHEAD=2 python tools/e2e_breakdown.py c3 60 20 8 > $O/e2e_breakdown_r4b_ahead2.txt 2>&1; head -7 $O/e2e_breakdown_r4b_ahead2.txt
timeout 600 python tools/self_collision_cost.py > $O/self_collision_cost_r4b.json 2>&1; cat $O/self_collision_cost_r4b.json
