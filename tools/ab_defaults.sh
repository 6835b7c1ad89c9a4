#!/bin/bash
# A/B of the candidate default switches on the headline workload (48M x 64 envs); run under gpurun
B="python bench.py --steps 200 --warmup 10 --no-cpu-baseline --profile-steps 0"
for o in "" "--opt l2_prefetch_mb=48" "--opt l2_prefetch_mb=96" "--opt state_impl=2" ""; do
  echo "== [$o]"
  timeout 120 $B $o "$@" 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.readline())
print(round(d['value']), round(d['e2e']['value']), round(d['ms_per_step']*1e3,1), 'us/step', d['clocks']['sm_mhz'])"
done
