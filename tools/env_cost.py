"""What environment lighting costs the render: M samples/s of rtx_render with the constant background, with a 1x1
map, and with a 4096x2048 map (128 MiB of float4 texels, larger than the B200's 126 MB L2), on the same resident scene.

A miss with a map evaluates E(d) of include/rttnw_b200.h: an f64 atan2 pair and a hypot, then four float4 loads. Scenes
1-4 end almost every path in a miss, scene 9 few. For each scene (at its default size, `--spp` samples per pixel) the
three settings are warmed up, then timed in `--reps` alternating rounds with CUDA events on the context's stream around
one synchronised call each. Prints the card's name and power limit first, then per setting the median and spread.

    python tools/env_cost.py            # scenes 1, 4 and 9, 128 spp
"""
import argparse
import os
import statistics
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rttnw_b200 as R  # noqa: E402
from tools.aov_cost import timed  # noqa: E402


def big_map(w, h, seed=1):
    """A smooth sky with a sun, so that neighbouring rays read neighbouring texels as a real HDRI would."""
    rng = np.random.default_rng(seed)
    v = ((np.arange(h, dtype=np.float32) + 0.5) / h)[:, None, None]
    u = ((np.arange(w, dtype=np.float32) + 0.5) / w)[None, :, None]
    img = 0.4 + 0.3 * np.sin(2 * np.pi * u * np.array([1, 2, 3], dtype=np.float32) + rng.random(3).astype(np.float32)) * np.sin(np.pi * v)
    img += 20.0 * np.exp(-(((u - 0.6) * 64) ** 2 + ((v - 0.3) * 64) ** 2))
    return np.ascontiguousarray(img, dtype=np.float32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", default="1,4,9")
    ap.add_argument("--spp", type=int, default=128)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    ctx = R.Context(0)
    large = big_map(4096, 2048)
    for n in map(int, args.scenes.split(",")):
        d = R.scene_defaults(n)
        w, h = d["width"], d["height"]
        gsc = R.DeviceScene(ctx, R.BuiltinDesc(n))
        one = np.array(R.BuiltinDesc(n).desc.background, dtype=np.float32).reshape(1, 1, 3)
        settings = {"background": None, "map 1x1": one, "map 4096x2048": large}
        accum = gsc.new_accum(w, h)

        def run():
            gsc.render_into(accum, 0, args.spp, seed=1, max_depth=d["max_depth"])

        times = {k: [] for k in settings}
        for k, m in settings.items():  # warm-up of every setting
            gsc.set_environment(m)
            timed(ctx, run)
        for _ in range(args.reps):
            for k, m in settings.items():
                gsc.set_environment(m)
                accum.zero_()
                times[k].append(timed(ctx, run))
        base = statistics.median(times["background"])
        for k, t in times.items():
            med = statistics.median(t)
            print(f"scene {n} {w}x{h} spp {args.spp}, {k}: {w * h * args.spp / med / 1e3:.1f} M samples/s, median {med:.2f} ms "
                  f"(min {min(t):.2f}, max {max(t):.2f}), {med / base:.3f} x the background's time, {args.reps} alternating reps",
                  flush=True)
        gsc.close()
    ctx.close()


if __name__ == "__main__":
    main()
