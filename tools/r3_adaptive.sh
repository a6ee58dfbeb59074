#!/bin/bash
# Round 3: adaptive sampling (rtx_render_adaptive) against uniform sampling, on the final scene at 800x800 and the Cornell
# box at 600x600 (tools/adaptive_quality.py), then bench.py on the default path with this build and, alternating, with
# the parent commit when a build of it is in old_lib/parent. Writes the log to stdout (profiles/r3_adaptive.txt).
cd "$(dirname "$0")/.."
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
for s in "9 800 800" "7 600 600"; do
  set -- $s
  echo "== tools/adaptive_quality.py --scene $1 --width $2 --height $3"
  timeout 1200 python tools/adaptive_quality.py --scene "$1" --width "$2" --height "$3" 2>&1
done
for rep in 1 2; do
  echo "== bench.py --gpus 1 --steps 8 --warmup 3 (this build, run $rep)"
  timeout 600 python bench.py --gpus 1 --steps 8 --warmup 3 --no-cpu-baseline 2>&1 | tail -1
  if [ -d old_lib/parent ]; then
    echo "== bench.py --gpus 1 --steps 8 --warmup 3 (the parent commit, built in old_lib/parent, run $rep)"
    (cd old_lib/parent && timeout 600 python bench.py --gpus 1 --steps 8 --warmup 3 --no-cpu-baseline 2>&1 | tail -1)
  fi
done
