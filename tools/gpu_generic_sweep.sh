#!/bin/bash
# A/B sweep of the generic locator's knobs on one B200: bucket fineness (RTHX_GRID_FINE) and bucket budget per face
# (RTHX_GRID_PER_FACE).  Prints rays/s per setting.
O=${1:-gpurun_out/sweep}; mkdir -p $O
run() {  # name workload env...
  local name=$1 w=$2; shift 2
  env "$@" timeout 200 python bench.py --workload $w --locator generic --steps 3 --warmup 2 --no-e2e --no-cpu-baseline --no-smoothing --no-extras --rays ${RAYS:-1e9} > $O/$name.json 2> $O/$name.err
  python - <<PY
import json
try:
    d=json.loads(open("$O/$name.json").read().strip().splitlines()[-1]); print("$name", "%.4g"%d["value"], "%.2f ms"%d["roofline"]["kernel_ms"], d["check"])
except Exception as e:
    print("$name", "FAILED", e)
PY
}
for w in cfg3 cfg5; do
  run ${w}_f8 $w RTHX_GRID_FINE=8
  run ${w}_f4 $w RTHX_GRID_FINE=4
  run ${w}_f6 $w RTHX_GRID_FINE=6
  run ${w}_f12 $w RTHX_GRID_FINE=12 RTHX_GRID_PER_FACE=200
  run ${w}_f16 $w RTHX_GRID_FINE=16 RTHX_GRID_PER_FACE=320
done
