#!/bin/bash
# Round 3: the denoiser (rtx_denoise). Its time against the 64-spp beauty pass and its quality against a 40 000-spp
# reference on the final scene at 800x800 and the Cornell box and the smoke box at 600x600, with the parameter sweep the
# defaults were chosen on (tools/denoise_quality.py), then bench.py on the default path with this build and,
# alternating, with the parent commit when a build of it is in old_lib/parent. Writes the log to stdout
# (profiles/r3_denoise.txt).
cd "$(dirname "$0")/.."
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
echo "== tools/denoise_quality.py --sweep"
timeout 1500 python tools/denoise_quality.py --sweep 2>&1
for rep in 1 2; do
  echo "== bench.py --gpus 1 --steps 8 --warmup 3 (this build, run $rep)"
  timeout 600 python bench.py --gpus 1 --steps 8 --warmup 3 --no-cpu-baseline 2>&1 | tail -1
  if [ -d old_lib/parent ]; then
    echo "== bench.py --gpus 1 --steps 8 --warmup 3 (the parent commit, built in old_lib/parent, run $rep)"
    (cd old_lib/parent && timeout 600 python bench.py --gpus 1 --steps 8 --warmup 3 --no-cpu-baseline 2>&1 | tail -1)
  fi
done
