"""What the feature-buffer pass (rtx_render_aov) costs next to the beauty pass (rtx_render) at equal spp.

For each (scene, size, spp): both calls on the same resident scene, warmed up, then `--reps` alternating repetitions,
each timed with CUDA events on the context's stream around one synchronised call (fresh zeroed buffers each time, kept
out of the window). Prints the card's name and power limit first, then per configuration the median and spread of both
times and their ratio.

    python tools/aov_cost.py            # scene 9 at 800x800 and scene 7 at 600x600, 64 and 256 spp
"""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rttnw_b200 as R  # noqa: E402


def timed(ctx, fn):
    torch = ctx.torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.sync()
    a.record(ctx.stream)
    fn()
    b.record(ctx.stream)
    ctx.sync()
    b.synchronize()
    return a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="9:800:800,7:600:600")
    ap.add_argument("--spp", default="64,256")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    ctx = R.Context(0)
    for cfg in args.configs.split(","):
        n, w, h = map(int, cfg.split(":"))
        depth = R.scene_defaults(n)["max_depth"]
        gsc = R.DeviceScene(ctx, R.BuiltinDesc(n))
        for spp in map(int, args.spp.split(",")):
            accum, aov = gsc.new_accum(w, h), gsc.new_aov(w, h)

            def beauty():
                gsc.render_into(accum, 0, spp, seed=1, max_depth=depth)

            def features():
                gsc.render_aov(aov, 0, spp, seed=1, max_depth=depth)

            for fn in (beauty, features):  # warm-up: module load, pool allocation
                timed(ctx, fn)
            tb, ta = [], []
            for _ in range(args.reps):
                accum.zero_()
                for t in aov.values():
                    t.zero_()
                tb.append(timed(ctx, beauty))
                ta.append(timed(ctx, features))
            mb, ma = statistics.median(tb), statistics.median(ta)
            print(f"scene {n} {w}x{h} spp {spp}: beauty {mb:.2f} ms (min {min(tb):.2f}, max {max(tb):.2f}), "
                  f"aov {ma:.2f} ms (min {min(ta):.2f}, max {max(ta):.2f}), aov / beauty {ma / mb:.3f}, "
                  f"aov {w * h * spp / ma / 1e3:.0f} M samples/s, {args.reps} alternating reps", flush=True)
        gsc.close()
    ctx.close()


if __name__ == "__main__":
    main()
