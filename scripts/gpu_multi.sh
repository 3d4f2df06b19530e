#!/bin/bash
# Multi-GPU evidence: fabric ceiling (all ranks copying at once), the multi-device engine tests, strong scaling of ONE
# engine over N devices, the torchrun bench line at N GPUs (both arms).
#   gpurun --gpus N --timeout 900 -- 'bash scripts/gpu_multi.sh <tag> N'
set -u
TAG=${1:-rXX}
N=${2:-2}
OUT=gpurun_out
mkdir -p $OUT
nvidia-smi --query-gpu=index,name,clocks.max.sm,memory.total --format=csv > $OUT/${TAG}_box_n$N.txt 2>&1
nproc >> $OUT/${TAG}_box_n$N.txt
nvidia-smi topo -m >> $OUT/${TAG}_box_n$N.txt 2>&1
TR="python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1"
timeout 300 $TR --master-port 29610 scripts/fabric_probe.py > $OUT/${TAG}_fabric_n$N.json 2> $OUT/${TAG}_fabric_n$N.err; tail -25 $OUT/${TAG}_fabric_n$N.json
timeout 600 python -m pytest tests -m gpu -x -q -k "devices or partitioner" > $OUT/${TAG}_pytest_multi_n$N.log 2>&1; tail -3 $OUT/${TAG}_pytest_multi_n$N.log
timeout 400 python scripts/multi_probe.py --max-devices $N > $OUT/${TAG}_multi_probe_shard_n$N.log 2>&1; tail -1 $OUT/${TAG}_multi_probe_shard_n$N.log | cut -c1-1500
timeout 600 $TR --master-port 29611 bench.py --impl reference --gpus $N --steps 2 --warmup 1 > $OUT/${TAG}_bench_ref_n$N.json 2> $OUT/${TAG}_bench_ref_n$N.err
tail -c 400 $OUT/${TAG}_bench_ref_n$N.json
timeout 600 $TR --master-port 29612 bench.py --gpus $N --steps 20 --warmup 3 > $OUT/${TAG}_bench_short8_n$N.json 2> $OUT/${TAG}_bench_short8_n$N.err
tail -c 1500 $OUT/${TAG}_bench_short8_n$N.json; tail -5 $OUT/${TAG}_bench_short8_n$N.err
python - <<PY
import json
try:
    d = json.loads(open("$OUT/${TAG}_bench_short8_n$N.json").read().strip().splitlines()[-1])
    print("e2e drop-in: %.1f GCUPS %.2f ms/step; packed %.1f GCUPS" % (d["e2e"]["value"], d["e2e"]["ms_per_step"], d["e2e"]["packed"]["value"]))
except Exception as e:
    print("no line", e)
PY
