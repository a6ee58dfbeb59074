"""What the denoiser (rtx_denoise) costs and buys.

Time: rtx_denoise alone at each configuration's size, the median of `--reps` calls timed with CUDA events on the
context's stream after a warm-up, against the 64-spp beauty pass (rtx_render, median of 5) of the same scene and size.

Quality: per scene a reference of `--ref-spp` uniform samples with another seed (2), then uniform frames at the ladder
`--ladder` (seed 1) and, at each of `--spp`, the denoised frame: the render split at spp / 2 (the accumulator copied
there), the feature pass of min(16, spp) samples and rtx_denoise at its defaults; plus one adaptive frame (max_spp =
the largest --spp, its aux as the half). Each frame's RMSE against the reference in 8-bit display units (256 *
clamp(sqrt(mean), 0, 0.999), kept in float, as tools/adaptive_quality.py) and its frame-mean signed difference (the
bias). Headline: the uniform spp, and seconds, the raw frame needs to reach each denoised RMSE, interpolated log-log
between ladder points, against what the denoised frame took (render + features + filter).

`--sweep` also filters every uniform --spp frame of every scene with a grid of parameter sets and prints each set's
geometric mean of denoised / raw RMSE over all of them: the one measurement the library's defaults were chosen on.

    python tools/denoise_quality.py                 # scene 9 at 800x800, scenes 7 and 8 at 600x600
"""
import argparse
import itertools
import math
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rttnw_b200 as R  # noqa: E402
from rttnw_b200.render import DENOISE_DEFAULTS  # noqa: E402


def display(x):
    import torch
    a = x.double()
    return 256.0 * torch.clamp(torch.sqrt(torch.clamp(a[..., :3] / a[..., 3:4], min=0.0)), 0.0, 0.999)


def events_ms(ctx, fn):
    torch = ctx.torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.sync()
    a.record(ctx.stream)
    fn()
    b.record(ctx.stream)
    ctx.sync()
    b.synchronize()
    return a.elapsed_time(b)


def wall(ctx, fn):
    ctx.sync()
    t0 = time.perf_counter()
    out = fn()
    ctx.sync()
    return time.perf_counter() - t0, out


def interp_loglog(pts, y):
    """x at which the piecewise log-log line through pts (x, y), y falling with x, reaches y; None outside."""
    pts = sorted(pts)
    for (x0, y0), (x1, y1) in zip(pts, pts[1:]):
        if min(y0, y1) <= y <= max(y0, y1) and y0 != y1:
            f = (math.log(y) - math.log(y0)) / (math.log(y1) - math.log(y0))
            return math.exp(math.log(x0) + f * (math.log(x1) - math.log(x0)))
    return None


SWEEP = {"iterations": (3, 4, 5, 6), "sigma_normal": (0.25, 0.5), "sigma_albedo": (0.1, 0.3),
         "sigma_luminance": (1.0, 2.0, 4.0, 8.0)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="9:800:800,7:600:600,8:600:600")
    ap.add_argument("--spp", default="16,64,256")
    ap.add_argument("--ladder", default="16,64,256,1024,4096")
    ap.add_argument("--ref-spp", type=int, default=40000)
    ap.add_argument("--adaptive", type=float, default=0.05, help="threshold of the adaptive frame")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--sweep", action="store_true")
    args = ap.parse_args()
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    spps = [int(s) for s in args.spp.split(",")]
    ladder = sorted(set(int(s) for s in args.ladder.split(",")) | set(spps))
    print(f"rtx_denoise defaults: {DENOISE_DEFAULTS}", flush=True)
    ctx = R.Context(0)
    sweep_rows = {}
    for cfg in args.configs.split(","):
        n, w, h = map(int, cfg.split(":"))
        depth = R.scene_defaults(n)["max_depth"]
        gsc = R.DeviceScene(ctx, R.BuiltinDesc(n))
        print(f"== scene {n} ({R.scene_defaults(n)['name']}) {w}x{h}", flush=True)
        acc, half, aov = gsc.new_accum(w, h), gsc.new_accum(w, h), gsc.new_aov(w, h)

        # ---- time
        def beauty():
            acc.zero_()
            gsc.render_into(acc, 0, 64, seed=1, max_depth=depth)

        beauty()
        half.copy_(acc)
        gsc.render_aov(aov, 0, 16, seed=1, max_depth=depth)
        ctx.denoise(acc, half, aov)  # warm-up
        tb = statistics.median(events_ms(ctx, beauty) for _ in range(5))
        td = [events_ms(ctx, lambda: ctx.denoise(acc, half, aov)) for _ in range(args.reps)]
        md = statistics.median(td)
        print(f"time: rtx_denoise {md:.3f} ms (min {min(td):.3f}, max {max(td):.3f}, {args.reps} calls) against the "
              f"64-spp beauty pass {tb:.2f} ms: {md / tb:.2%}", flush=True)

        # ---- reference and raw ladder
        ref = gsc.new_accum(w, h)
        dt, _ = wall(ctx, lambda: gsc.render_into(ref, 0, args.ref_spp, seed=2, max_depth=depth))
        ref_d = display(ref)
        del ref
        print(f"reference: {args.ref_spp} spp, seed 2, {dt:.2f} s", flush=True)

        def score(x):
            d = display(x)
            return float(((d - ref_d) ** 2).mean().sqrt()), float((d - ref_d).mean())

        raw_pts, raw_secs = [], {}
        for spp in ladder:
            acc.zero_()
            dt, _ = wall(ctx, lambda: gsc.render_into(acc, 0, spp, seed=1, max_depth=depth))
            rm, ms = score(acc)
            raw_pts.append((spp, rm))
            raw_secs[spp] = dt
            print(f"raw      {spp:6d} spp: {dt:7.3f} s, RMSE {rm:8.4f}, mean signed {ms:+.4f}", flush=True)

        def denoised_row(label, render_s, feat_spp, half_buf):
            aov_ = gsc.new_aov(w, h)
            tf, _ = wall(ctx, lambda: gsc.render_aov(aov_, 0, feat_spp, seed=1, max_depth=depth))
            tdn, out = wall(ctx, lambda: ctx.denoise(acc, half_buf, aov_))
            rm_raw, ms_raw = score(acc)
            rm, ms = score(out)
            total = render_s + tf + tdn
            need = interp_loglog(raw_pts, rm)
            need_s = interp_loglog([(raw_secs[s], r) for s, r in raw_pts], rm)
            lo, hi = min(raw_pts), max(raw_pts)
            print(f"{label}: raw RMSE {rm_raw:8.4f} (mean signed {ms_raw:+.4f}) -> denoised {rm:8.4f} (mean signed "
                  f"{ms:+.4f}), ratio {rm / rm_raw:.3f}; render {render_s:.3f} s + features ({feat_spp} spp) {tf:.3f} s "
                  f"+ filter {tdn * 1e3:.1f} ms = {total:.3f} s; raw needs "
                  + (f"{need:.0f} spp / {need_s:.3f} s for that RMSE: {need_s / total:.2f}x the time"
                     if need else (f"more than {hi[0]} spp for that RMSE" if rm < hi[1] else
                                   f"no more than {lo[0]} spp for that RMSE: no gain")),
                  flush=True)
            return aov_

        for spp in spps:
            acc.zero_()
            ctx.sync()
            t0 = time.perf_counter()
            gsc.render_into(acc, 0, spp // 2, seed=1, max_depth=depth)
            half.copy_(acc)
            gsc.render_into(acc, spp // 2, spp - spp // 2, seed=1, max_depth=depth)
            ctx.sync()
            aov_s = denoised_row(f"uniform  {spp:6d} spp", time.perf_counter() - t0, min(16, spp), half)
            if args.sweep:
                for combo in itertools.product(*SWEEP.values()):
                    p = dict(zip(SWEEP, combo))
                    rm, _ = score(ctx.denoise(acc, half, aov_s, **p))
                    sweep_rows.setdefault(combo, []).append(rm / score(acc)[0])
        mx = max(spps)
        mn = max(2, (mx // 64 + 1) // 2 * 2)
        dt, st = wall(ctx, lambda: gsc.render_adaptive(acc, half, args.adaptive, mn, mn, mx, seed=1, max_depth=depth))
        denoised_row(f"adaptive {args.adaptive} (min {mn}, max {mx}, {st['path_samples'] / (w * h):.1f} spp mean)", dt,
                     min(16, mx), half)
        gsc.close()
    if args.sweep:
        print(f"== sweep: geometric mean of denoised / raw RMSE over the {len(next(iter(sweep_rows.values())))} uniform "
              "frames, best first")
        ranked = sorted(sweep_rows.items(), key=lambda kv: sum(math.log(r) for r in kv[1]))
        for combo, rs in ranked[:12]:
            g = math.exp(sum(math.log(r) for r in rs) / len(rs))
            print(f"  {dict(zip(SWEEP, combo))}: {g:.4f} (worst {max(rs):.3f})")
        d = (5, 0.25, 0.1, 4.0)
        g = math.exp(sum(math.log(r) for r in sweep_rows[d]) / len(sweep_rows[d]))
        print(f"  the starting point {dict(zip(SWEEP, d))}: {g:.4f} (worst {max(sweep_rows[d]):.3f})")
    ctx.close()


if __name__ == "__main__":
    main()
