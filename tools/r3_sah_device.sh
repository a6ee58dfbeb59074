#!/bin/bash
# Round 3: the device binned-SAH builder (RTX_BVH=sah_device) against host SAH, LBVH and PLOC. Build time, node
# visits per ray and trace rate on 2e5, 1e6 and 2e6 random spheres (host SAH up to 1e6), then renders of scenes 9 and 1
# with the host-built and the device-built tree, alternating. Writes the log to stdout (profiles/r3_sah_device.txt).
cd "$(dirname "$0")/.."
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
for n in 200000 1000000 2000000; do
  echo "== tools/big_scene.py $n"
  RTX_DEBUG_BUILD=1 timeout 900 python tools/big_scene.py $n 2>&1
done
for s in 9 1; do
  echo "== tools/quick_ab.py --scene $s"
  timeout 600 python tools/quick_ab.py --scene $s --spp 128 --reps 3 "RTX_BVH=sah" "RTX_BVH=sah_device" "RTX_BVH=sah" "RTX_BVH=sah_device" 2>&1
done
