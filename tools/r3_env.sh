#!/bin/bash
# Round 3: environment lighting (rtx_scene_set_environment). Its cost on scenes 1, 4 and 9 at their default sizes and
# 128 spp with the background, a 1x1 map and a 4096x2048 map (tools/env_cost.py), then bench.py on the default path
# with this build and, alternating, with the parent commit when a build of it is in old_lib/parent. Writes the log to
# stdout (profiles/r3_env.txt).
cd "$(dirname "$0")/.."
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
echo "== tools/env_cost.py"
timeout 1200 python tools/env_cost.py 2>&1
for rep in 1 2; do
  echo "== bench.py --gpus 1 --steps 8 --warmup 3 (this build, run $rep)"
  timeout 600 python bench.py --gpus 1 --steps 8 --warmup 3 --no-cpu-baseline 2>&1 | tail -1
  if [ -d old_lib/parent ]; then
    echo "== bench.py --gpus 1 --steps 8 --warmup 3 (the parent commit, built in old_lib/parent, run $rep)"
    (cd old_lib/parent && timeout 600 python bench.py --gpus 1 --steps 8 --warmup 3 --no-cpu-baseline 2>&1 | tail -1)
  fi
done
