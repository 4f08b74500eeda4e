# 2 GPUs: the two routes of the gradient all-reduce (correctness through tools/dist_check.py, then the bench line)
TR="python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1"
mkdir -p gpurun_out
P=29520
for v in "ctx:CTXNERF_NCCL=1" "torch:CTXNERF_NCCL=0"; do
  name=${v%%:*}; envs=${v#*:}
  env $envs timeout 300 $TR --master-port $P tools/dist_check.py > gpurun_out/dist2_$name.log 2>&1; echo "dist_check $name rc=$?"; P=$((P+1))
  if [ "$1" = "bench" ]; then
    env $envs timeout 400 $TR --master-port $P bench.py --gpus 2 --steps 20 --warmup 5 --no-sustained > gpurun_out/bench2_$name.log 2>&1; echo "bench $name rc=$?"; P=$((P+1))
    tail -1 gpurun_out/bench2_$name.log | python -c "import json,sys; d=json.loads(sys.stdin.read()); print(d['value'], d['ms_per_step'], d['e2e']['value'], d.get('allreduce'))"
  fi
  grep -h "^rank" gpurun_out/dist2_$name.log
done
