#!/bin/bash
# Round 3: the feature-buffer pass (rtx_render_aov). Its cost against the beauty pass at equal spp on the final scene at
# 800x800 and the Cornell box at 600x600 (tools/aov_cost.py), then bench.py on the default path with this build and,
# alternating, with the parent commit when a build of it is in old_lib/parent. Writes the log to stdout
# (profiles/r3_aov.txt).
cd "$(dirname "$0")/.."
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
echo "== tools/aov_cost.py"
timeout 900 python tools/aov_cost.py 2>&1
for rep in 1 2; do
  echo "== bench.py --gpus 1 --steps 8 --warmup 3 (this build, run $rep)"
  timeout 600 python bench.py --gpus 1 --steps 8 --warmup 3 --no-cpu-baseline 2>&1 | tail -1
  if [ -d old_lib/parent ]; then
    echo "== bench.py --gpus 1 --steps 8 --warmup 3 (the parent commit, built in old_lib/parent, run $rep)"
    (cd old_lib/parent && timeout 600 python bench.py --gpus 1 --steps 8 --warmup 3 --no-cpu-baseline 2>&1 | tail -1)
  fi
done
