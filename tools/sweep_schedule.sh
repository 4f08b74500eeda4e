#!/bin/bash
# bench.py under several backward schedules / SM budgets (one JSON line each -> gpurun_out/sweep_schedule.txt)
out=gpurun_out/sweep_schedule.txt
: > $out
run() { echo "== $*" >> $out; env "$@" python bench.py --steps 20 --warmup 3 --no-cpu-baseline 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1])
g=(d['roofline'] or {}).get('concurrent_group') or {}
print(round(d['ms_per_step'],4), round(d['value']), 'e2e', round(d['e2e']['ms_per_step'],4), 'group', g.get('ms'))" >> $out; }
run CTXNERF_SIDE_SMS=44
run CTXNERF_SIDE_SMS=36
run CTXNERF_SIDE_SMS=52
run CTXNERF_SIDE_SMS=60
run CTXNERF_SIDE_SMS=28
run CTXNERF_OVERLAP=0
run CTXNERF_GRAPH=0
cat $out
