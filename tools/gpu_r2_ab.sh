#!/bin/bash
# interleaved same-box A/B of step-level switches (the chip runs at its power cap: single runs drift by ~2 %)
mkdir -p gpurun_out
S="--steps 20 --warmup 5 --no-eager --no-cpu-baseline --no-aux"
: > gpurun_out/r2_ab.log
for rep in 1 2 3; do
  for cfg in "1 1" "0 1" "1 0"; do
    set -- $cfg
    export J="$(HDRVAE_FUSE_NIN=$1 HDRVAE_H16=$2 timeout 600 python bench.py $S | tail -1)"
    python - >> gpurun_out/r2_ab.log <<PY
import json, os
d = json.loads(os.environ["J"])
print("rep $rep nin=$1 h16=$2", round(d["ms_per_step"], 3), "ms", round(d["value"], 2), "MP/s  clock", d["clocks"]["sm_mhz"], d["roofline"]["step_breakdown_ms"])
PY
  done
done
cat gpurun_out/r2_ab.log
