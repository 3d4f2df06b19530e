#!/bin/bash
# SM clock while global_bench runs (bursts of 2-3 ms of GPU work every ~7 ms)
T=${1:-r04c}
mkdir -p gpurun_out
nvidia-smi --query-gpu=clocks.sm,clocks.mem,power.draw,clocks_throttle_reasons.active --format=csv,noheader -lms 50 > gpurun_out/${T}_clocks.csv 2>&1 &
SMI=$!
BSW_GLOBAL_CHUNK=262144 GLOBAL_BENCH_NO_CPU=1 timeout 60 python scripts/global_bench.py 300 150 > gpurun_out/${T}_global_bench_k2_chunk262144_reps150.json 2>&1
kill $SMI
sort gpurun_out/${T}_clocks.csv | uniq -c | sort -rn | head -8
