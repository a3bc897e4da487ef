#!/bin/bash
# A/B runs of the multi-GPU path on N GPUs of one box (under gpurun --gpus N): tests, bench with trace, switches off one by one.
# usage: scripts/run_mgpu_ab.sh N tag [notests]
N=$1; TAG=$2
TR="python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1"
if [ "$3" != "notests" ]; then
  python -m pytest tests -m gpu -x -q > gpurun_out/${TAG}_tests.log 2>&1; echo "pytest rc=$?" >> gpurun_out/${TAG}_tests.log
fi
$TR --master-port 29601 bench.py --gpus $N --steps 5 --warmup 3 --trace gpurun_out/${TAG}_trace_full > gpurun_out/${TAG}_bench_full.json 2> gpurun_out/${TAG}_bench_full.err; echo "rc=$?" >> gpurun_out/${TAG}_bench_full.err
P=29602
for SW in "PAMG_FOLD_CHECK=0"; do
  NAME=$(echo "$SW" | tr ' =' '__')
  env $SW $TR --master-port $P bench.py --gpus $N --steps 5 --warmup 3 --no-cpu-baseline --no-small-parity --secondary none \
      --trace gpurun_out/${TAG}_trace_${NAME} > gpurun_out/${TAG}_bench_${NAME}.json 2> gpurun_out/${TAG}_bench_${NAME}.err; echo "rc=$?" >> gpurun_out/${TAG}_bench_${NAME}.err
  P=$((P+1))
done
tail -3 gpurun_out/${TAG}_tests.log 2>/dev/null
for f in gpurun_out/${TAG}_bench_*.json; do echo $f; python -c "
import json,sys
try:
    d=json.loads(open('$f').read().strip().splitlines()[-1]); print(d['ms_per_step'], d['config']['iters'], d['e2e']['ms_per_step'], d.get('parity'))
except Exception as e: print('ERR', e)
"; done
tail -2 gpurun_out/${TAG}_bench_*.err
