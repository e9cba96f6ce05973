#!/bin/bash
# A/B of steps in flight on one B200, alternating
B="python bench.py --no-cpu-baseline --no-eager-baseline --steps 100"
for rep in 1 2 3; do
  for ov in 4 5 6 8; do
    v=$($B --overlap $ov 2>/dev/null | python -c "import json,sys; d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print(round(d['value']), d['ms_per_step'])")
    echo "rep $rep overlap $ov: $v"
  done
done
