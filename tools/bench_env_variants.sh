#!/bin/bash
# bench.py under several environment settings, one summary line each
run() { env "$@" timeout 200 python bench.py --steps 20 --warmup 5 --no-cpu-baseline --no-sustained 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1])
print('$*', round(d['value']), round(d['ms_per_step'],4), round(d['e2e']['ms_per_step'],4), round(d['step_tensor_frac'],4))
"; }
for rep in 1 2; do
run X=0
run CTXNERF_OVERLAP=0
run CTXNERF_SIDE_SMS=52
done
