"""Does adaptive sampling reach a given image quality sooner than uniform sampling? (rtx_render_adaptive)

For one scene: a reference frame (uniform, another seed, 4x the largest spp compared), then uniform renders at the
given spp and adaptive renders at four thresholds, each timed end to end (host clock around a synchronised call, the
scene already resident and the kernels warmed up). For every frame: RMSE against the reference in 8-bit display units
(256 * clamp(sqrt(mean), 0, 0.999), main.rs:217-225, kept in float), wall time, path samples and samples/s; for the
adaptive ones also the rounds, the frame-mean signed difference against the reference per class of tile count (at
min_spp, in between, at max_spp) and, from a second run with RTX_DEBUG_ADAPTIVE=1, the rate of every round.

The thresholds are derived from the frame itself: the tile errors of a min_spp frame, scaled by sqrt(min_spp / max_spp)
(the error of a mean falls as 1 / sqrt(n)), predict each tile's error at max_spp; the thresholds are the 10th, 30th,
50th and 80th percentiles of that prediction. The RMSE includes the reference's own noise (a quarter of the variance of
the largest uniform frame), which is the same for every frame compared.

    python tools/adaptive_quality.py --scene 9 --width 800 --height 800
"""
import argparse
import json
import math
import os
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rttnw_b200 as R  # noqa: E402


def display(acc):
    import torch
    a = acc.double()
    return 256.0 * torch.clamp(torch.sqrt(torch.clamp(a[..., :3] / a[..., 3:4], min=0.0)), 0.0, 0.999)


def rmse(d, ref_d):
    return float(((d - ref_d) ** 2).mean().sqrt())


class StderrLines:
    """Collects what the library writes to fd 2 inside the block."""

    def __enter__(self):
        sys.stderr.flush()
        self.tmp = tempfile.TemporaryFile(mode="w+b")
        self.saved = os.dup(2)
        os.dup2(self.tmp.fileno(), 2)
        return self

    def __exit__(self, *exc):
        sys.stderr.flush()
        os.dup2(self.saved, 2)
        os.close(self.saved)
        self.tmp.seek(0)
        self.lines = self.tmp.read().decode().splitlines()
        self.tmp.close()


def parse_round(line):
    # "[rtx] adaptive round R: T tiles x S spp (n = N), P path samples, render X ms[, decision Y ms]"
    parts = line.replace(",", "").split()
    vals = {"round": int(parts[3].rstrip(":")), "tiles": int(parts[4]), "spp": int(parts[7]), "n": int(parts[11].rstrip(")")),
            "path_samples": int(parts[12]), "render_ms": float(parts[16])}
    vals["decision_ms"] = float(parts[19]) if len(parts) > 19 else 0.0
    return vals


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scene", type=int, default=9)
    ap.add_argument("--width", type=int, default=800)
    ap.add_argument("--height", type=int, default=800)
    ap.add_argument("--spp", default="256,1024,4096,10000", help="uniform spp compared; the largest is max_spp")
    ap.add_argument("--quantiles", default="0.1,0.3,0.5,0.8")
    ap.add_argument("--json", default="")
    args = ap.parse_args()
    import torch
    spps = [int(s) for s in args.spp.split(",")]
    max_spp = max(spps)
    min_spp = max(2, (max_spp // 64 + 1) // 2 * 2)
    w, h = args.width, args.height
    d = R.scene_defaults(args.scene)
    depth = d["max_depth"]
    ctx = R.Context(0)
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(args.scene))
    out = {"scene": args.scene, "width": w, "height": h, "max_depth": depth, "min_spp": min_spp, "step_spp": min_spp,
           "max_spp": max_spp, "uniform": [], "adaptive": []}
    print(f"scene {args.scene} ({d['name']}) {w}x{h}, depth {depth}; adaptive min_spp = step_spp = {min_spp}, max_spp = {max_spp}", flush=True)

    # warm-up: module load, pool allocation
    acc = gsc.new_accum(w, h)
    aux = gsc.new_accum(w, h)
    gsc.render_into(acc, 0, 8, seed=1, max_depth=depth)
    gsc.render_adaptive(acc, aux, 0.0, 2, 2, 4, seed=1, max_depth=depth)
    ctx.sync()

    ref_spp = 4 * max_spp
    ref = gsc.new_accum(w, h)
    t0 = time.perf_counter()
    gsc.render_into(ref, 0, ref_spp, seed=2, max_depth=depth)
    ctx.sync()
    print(f"reference: {ref_spp} spp, seed 2, {time.perf_counter() - t0:.2f} s", flush=True)
    ref_d = display(ref)
    del ref

    for spp in spps:
        acc.zero_()
        ctx.sync()
        t0 = time.perf_counter()
        gsc.render_into(acc, 0, spp, seed=1, max_depth=depth)
        ctx.sync()
        dt = time.perf_counter() - t0
        dd = display(acc)
        row = {"spp": spp, "seconds": dt, "path_samples": spp * w * h, "samples_per_s": spp * w * h / dt,
               "rmse": rmse(dd, ref_d), "mean_signed": float((dd - ref_d).mean())}
        out["uniform"].append(row)
        print(f"uniform  {spp:6d} spp: {dt:8.3f} s, {row['samples_per_s'] / 1e6:7.1f} M samples/s, RMSE {row['rmse']:.4f}, "
              f"mean signed {row['mean_signed']:+.4f}", flush=True)

    # thresholds from the min_spp frame's tile errors, projected to max_spp
    gsc.render_adaptive(acc, aux, 0.0, min_spp, min_spp, min_spp, seed=1, max_depth=depth)
    e = gsc.adaptive_error(acc, aux).cpu().numpy().astype(np.float64) * math.sqrt(min_spp / max_spp)
    thresholds = [float(np.quantile(e, float(q))) for q in args.quantiles.split(",")]
    print("thresholds (percentiles " + args.quantiles + " of the projected max_spp tile error): "
          + ", ".join(f"{t:.5g}" for t in thresholds), flush=True)

    for thr in thresholds:
        ctx.sync()
        t0 = time.perf_counter()
        st = gsc.render_adaptive(acc, aux, thr, min_spp, min_spp, max_spp, seed=1, max_depth=depth)
        dt = time.perf_counter() - t0
        dd = display(acc)
        n = acc[..., 3]
        classes = {"at_min": n == min_spp, "between": (n > min_spp) & (n < max_spp), "at_max": n == max_spp}
        bias = {}
        for k, m in classes.items():
            cnt = int(m.sum())
            bias[k] = {"pixels": cnt, "mean_signed": float((dd - ref_d)[m].mean()) if cnt else None,
                       "rmse": float(((dd - ref_d)[m] ** 2).mean().sqrt()) if cnt else None}
        os.environ["RTX_DEBUG_ADAPTIVE"] = "1"
        with StderrLines() as cap:
            gsc.render_adaptive(acc, aux, thr, min_spp, min_spp, max_spp, seed=1, max_depth=depth)
        del os.environ["RTX_DEBUG_ADAPTIVE"]
        rounds = [parse_round(l) for l in cap.lines if l.startswith("[rtx] adaptive round")]
        for r in rounds:
            r["samples_per_s"] = r["path_samples"] / (r["render_ms"] * 1e-3) if r["render_ms"] > 0 else 0.0
        row = {"threshold": thr, "seconds": dt, "path_samples": st["path_samples"], "samples_per_s": st["path_samples"] / dt,
               "spp_mean": st["path_samples"] / (w * h), "rounds": st["rounds"], "tiles": st["tiles"],
               "tiles_converged": st["tiles_converged"], "tiles_at_max": st["tiles_at_max"], "rmse": rmse(dd, ref_d),
               "mean_signed": float((dd - ref_d).mean()), "by_class": bias, "round_log": rounds}
        out["adaptive"].append(row)
        print(f"adaptive {thr:.5g}: {dt:8.3f} s, {row['spp_mean']:8.1f} spp mean, {row['samples_per_s'] / 1e6:7.1f} M samples/s, "
              f"{st['rounds']} rounds, {st['tiles_converged']}/{st['tiles']} tiles converged, RMSE {row['rmse']:.4f}, "
              f"mean signed {row['mean_signed']:+.4f}", flush=True)
        for k, b in bias.items():
            if b["pixels"]:
                print(f"    {k:8s}: {b['pixels']:8d} pixels, mean signed {b['mean_signed']:+.4f}, RMSE {b['rmse']:.4f}")
        for r in rounds:
            print(f"    round {r['round']:3d}: {r['tiles']:7d} tiles x {r['spp']:5d} spp, render {r['render_ms']:9.2f} ms "
                  f"({r['samples_per_s'] / 1e6:7.1f} M samples/s), decision {r['decision_ms']:6.2f} ms")
        late = [r for r in rounds if r["tiles"] <= 0.1 * st["tiles"]]
        if late:
            ps = sum(r["path_samples"] for r in late)
            ms = sum(r["render_ms"] for r in late)
            print(f"    late rounds (<= 10 % of tiles active): {len(late)}, {ps / (ms * 1e-3) / 1e6:.1f} M samples/s over {ms:.1f} ms")
        sys.stdout.flush()

    # headline: the time each method needs to reach the RMSE of the uniform max_spp frame (log-log interpolation)
    target = out["uniform"][-1]["rmse"]

    def time_to(rows):
        pts = sorted((r["rmse"], r["seconds"]) for r in rows)
        for (r0, t0), (r1, t1) in zip(pts, pts[1:]):
            if r0 <= target <= r1 and r1 > r0:
                f = (math.log(target) - math.log(r0)) / (math.log(r1) - math.log(r0))
                return math.exp(math.log(t0) + f * (math.log(t1) - math.log(t0)))
        return None

    # ... and, the other way round, the time uniform sampling needs for each adaptive frame's RMSE
    for row in out["adaptive"]:
        target_row = row["rmse"]
        pts = sorted((r["rmse"], r["seconds"]) for r in out["uniform"])
        row["uniform_seconds_for_this_rmse"] = None
        for (r0, t0), (r1, t1) in zip(pts, pts[1:]):
            if r0 <= target_row <= r1 and r1 > r0:
                f = (math.log(target_row) - math.log(r0)) / (math.log(r1) - math.log(r0))
                row["uniform_seconds_for_this_rmse"] = math.exp(math.log(t0) + f * (math.log(t1) - math.log(t0)))
        u = row["uniform_seconds_for_this_rmse"]
        print(f"adaptive {row['threshold']:.5g}: RMSE {row['rmse']:.4f} in {row['seconds']:.3f} s; uniform needs "
              + (f"{u:.3f} s for it ({row['seconds'] / u - 1:+.1%})" if u else "a time outside the measured range"))
    out["target_rmse"] = target
    out["uniform_seconds_to_target"] = out["uniform"][-1]["seconds"]
    out["adaptive_seconds_to_target"] = time_to(out["adaptive"])
    a = out["adaptive_seconds_to_target"]
    print(f"headline: RMSE of uniform {max_spp} spp = {target:.4f}; uniform reaches it in {out['uniform_seconds_to_target']:.3f} s, "
          + (f"adaptive in {a:.3f} s (interpolated between thresholds)" if a else
             "adaptive does not reach it at any threshold tried (no interpolation possible)"), flush=True)
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)
    gsc.close()
    ctx.close()


if __name__ == "__main__":
    main()
