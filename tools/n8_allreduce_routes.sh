#!/bin/bash
# N GPUs: the bench line under the two routes of the gradient all-reduce, twice each (run-to-run noise)
N=${1:-8}
TR="timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1"
P=29530
for rep in 1 2; do
for v in "ctx:CTXNERF_NCCL=1" "torch:CTXNERF_NCCL=0"; do
  name=${v%%:*}; envs=${v#*:}
  env $envs $TR --master-port $P bench.py --gpus $N --steps 20 --warmup 5 --no-sustained 2>/dev/null | tail -1 > gpurun_out/bench${N}_${name}_$rep.json; P=$((P+1))
  python -c "import json; d=json.load(open('gpurun_out/bench${N}_${name}_$rep.json')); print('$name', $rep, round(d['ms_per_step'],4), round(d['value']), round(d['e2e']['value']))"
done
done
