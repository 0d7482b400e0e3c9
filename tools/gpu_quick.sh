#!/bin/bash
# Short GPU-box visit while iterating on a kernel: parity tests + the device/e2e bench line (no CPU leg, no ncu).
# usage (on the GPU box): bash tools/gpu_quick.sh [tag]
set -u
TAG=${1:-quick}
OUT=gpurun_out/$TAG
mkdir -p $OUT
( timeout 900 python -m pytest tests -m gpu -x -q 2>&1 | tail -15 ) > $OUT/pytest_gpu.log
( timeout 600 python bench.py --steps 10 --warmup 3 --no-cpu 2> $OUT/bench.err | tail -1 ) > $OUT/bench.json
tail -3 $OUT/pytest_gpu.log
python - <<PY
import json
d = json.load(open("$OUT/bench.json"))
print("value %.1f M atoms/s  e2e %.1f  ms/step %.3f" % (d["value"] / 1e6, d["e2e"]["value"] / 1e6, d["ms_per_step"]))
PY
