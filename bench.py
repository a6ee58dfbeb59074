#!/usr/bin/env python
"""bench.py — path samples/s of the rttnw hot path on the book-2 final scene (scene 9, 800x800).

A "step" is one pass of the hot path over one batch: every rank renders `--spp` samples per
pixel of the whole 800x800 frame (distinct global sample indices per rank and step), the
per-rank fp32 accumulators are combined on rank 0 and tonemapped to RGBA8. Samples are i.i.d.
(src/main.rs:211-217), so the path shards by spp with no data-path collective except that
end-of-frame combine; per-GPU work is fixed as N grows ("weak").

  value : W*H*spp*N*K / T, scene resident in HBM, T from CUDA events (max over ranks)
  e2e   : the same metric through the public API with HOST buffers: every step uploads the scene
          description (rtx_scene_create: H2D), renders, combines, tonemaps and reads the RGBA8
          frame back to the host (D2H) inside the timed region
  frames : the jobs BASELINE.json's metric names, timed once each with the same barrier / event bracket — `final_10k`
          (scene 9, 800x800, 10 000 spp IN TOTAL, split over the N ranks: STRONG scaling, efficiency = T(1) / (N T(N)))
          and `cornell_box` / `cornell_smoke` (scenes 7 and 8, 600x600, --cornell-spp in total)
  --impl reference : the reference's own CPU implementation of the path (the C++ f64 oracle — the
          Rust reference cannot be built here), all host threads, on a bounded sample of the frame
  --dump-outputs DIR : (GPU arm) what the last timed step computed, as .npy files: the same arguments give the same
          samples on every run, so two builds can be compared output for output
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SCENE = 9
METRIC = "path samples/sec"
UNIT = "samples/s"
# the scene table of src/main.rs:66-183 (width, height, samples per pixel, max depth, name), for the CPU arm, which must
# not load the product library; the GPU arm checks it against rtx_builtin_scene_defaults
SCENE_TABLE = {1: (400, 225, 100, 50, "random_scene"), 2: (400, 225, 100, 50, "two_spheres"), 3: (400, 225, 100, 50, "two_perlin_spheres"),
               4: (400, 225, 100, 50, "earth"), 5: (400, 225, 400, 50, "simple_light"), 6: (600, 600, 200, 50, "empty_cornell_box"),
               7: (600, 600, 200, 50, "cornell_box"), 8: (600, 600, 200, 50, "smoke_cornell_box"), 9: (800, 800, 10000, 50, "final_scene")}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--spp", type=int, default=128, help="samples per pixel per rank per step")
    ap.add_argument("--scene", type=int, default=SCENE)
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--combine", default="auto", choices=["auto", "peer", "slice", "nccl"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU work for the baseline sample")
    ap.add_argument("--no-frames", action="store_true", help="skip the final_10k / Cornell frames")
    ap.add_argument("--big-scene", type=int, default=2_000_000, help="spheres of the out-of-cache closest-hit leg at N=1 (0: skip)")
    ap.add_argument("--final-spp", type=int, default=10000, help="total spp of the final_10k frame (the reference default)")
    ap.add_argument("--cornell-spp", type=int, default=8000, help="total spp of the Cornell frames (reference default 200: too short to time)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed on rank 0 to DIR/<name>.npy (float32): `accum`, the (H, W, 4) "
                         "fp32 accumulator after the combine, and `frame`, the (H, W, 4) RGBA8 frame; past 64 MB in all, the same "
                         "seeded sample of pixels from both, with their flat indices in `pixel_index`")
    return ap.parse_args()


def scene_defaults(number):
    w, h, spp, depth, name = SCENE_TABLE[number]
    return {"width": w, "height": h, "samples": spp, "max_depth": depth, "name": name}


def workload(args):
    d = scene_defaults(args.scene)
    w, h = args.width or d["width"], args.height or d["height"]
    return d, w, h


def kernels_sha():
    """Hash of the kernel sources: the committed ncu counters are only used when they belong to the sources that run."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "rttnw_b200", "csrc")
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cuh", ".h", ".hpp", ".cpp")) and name not in ("cli.cpp", "png_io.cpp"):  # (what shapes the kernels' work)
            h.update(name.encode())
            h.update(open(os.path.join(d, name), "rb").read())
    return h.hexdigest()[:16]


def load_counters(scene):
    """profiles/r2_counters_s<scene>.json (tools/r2_profile.sh + tools/r2_counters.py): warp instructions, lanes, DRAM
    and L2 bytes PER PATH SAMPLE of each wavefront kernel, summed over every launch of one render under ncu. Per-sample
    counts are a property of the build and the scene, not of the run, so they combine with this run's measured
    samples/s into live rates. A file that was captured on other kernel sources is refused."""
    path = os.path.join(ROOT, "profiles", f"r2_counters_s{scene}.json")
    try:
        doc = json.load(open(path))
    except Exception as e:  # noqa: BLE001
        return None, f"no counters on file ({e})"
    if doc.get("kernels_sha") != kernels_sha():
        return None, f"{os.path.basename(path)} was captured on kernel sources {doc.get('kernels_sha')}, these are {kernels_sha()}: re-run tools/r2_profile.sh"
    return doc, None


def issue_roof(counters, samples_per_s, clocks, sms):
    """Warp instructions issued per second (instructions per path sample from the ncu counters x this run's measured
    path samples/s) against the SMs' issue slots at the SM clock sampled during the timed region: the roof SURVEY.md
    §8d names first for this path. Also the warp-execution efficiency (lanes per warp instruction / 32)."""
    mhz = (clocks or {}).get("sm_mhz") or 1965.0
    per_sample = sum(k["warp_instructions_per_sample"] for k in counters["kernels"].values())
    achieved = per_sample * samples_per_s / 1e9
    peak = 4.0 * sms * mhz * 1e6 / 1e9
    out = {"achieved": achieved, "peak": peak, "unit": "G warp instructions/s", "frac": achieved / peak,
           "warp_instructions_per_sample": per_sample, "sm_mhz": mhz, "sms": sms, "kernels": {}}
    for name, k in counters["kernels"].items():
        out["kernels"][name] = {"warp_instructions_per_sample": k["warp_instructions_per_sample"],
                                "lanes_per_warp_instruction": k["lanes_per_warp_instruction"],
                                "warp_execution_efficiency": k["lanes_per_warp_instruction"] / 32.0,
                                "instructions_per_active_sm_cycle_alone": k["instructions_per_active_sm_cycle"]}
    return out


def config(args, d, w, h):
    """The workload, and nothing else: both arms print the same dict (arm-specific facts go to `details`)."""
    return {"workload": f"scene {args.scene} ({d['name']}) {w}x{h}, max depth {d['max_depth']}, "
                        f"{args.spp} spp per GPU per step; reference default is {d['samples']} spp per frame",
            "scene": args.scene, "width": w, "height": h, "spp_per_gpu_per_step": args.spp,
            "max_depth": d["max_depth"], "sharding": "samples per pixel across GPUs, one combine per step",
            "l2": "flushed between timed steps (256 MiB write); the scene working set itself is L2-resident by nature"}


# ---------------------------------------------------------------------------
# CPU legs (the oracle is the checker / the reported baseline, never the product)
# ---------------------------------------------------------------------------
def oracle_scene(scene):
    import numpy as np
    from PIL import Image
    from tests import _oracle as O
    earth = np.ascontiguousarray(np.asarray(Image.open(os.path.join(ROOT, "assets", "earth.png")).convert("RGBA"), dtype=np.uint8))
    t0 = time.perf_counter()
    osc = O.OracleScene.builtin(scene, earth=earth)  # scene construction incl. the reference's own BVH build (Q17)
    return O, osc, time.perf_counter() - t0


def cpu_sample(osc, w, h, max_depth, stride, spp, seed, threads):
    t0 = time.perf_counter()
    _, rays = osc.render_sum(w, h, spp, seed=seed, max_depth=max_depth, rows=(stride // 2, h), row_stride=stride, threads=threads)
    dt = time.perf_counter() - t0
    rows = len(range(stride // 2, h, stride))
    return rows * w * spp, rays, dt


def cpu_scene_leg(scene, seconds, width=0, height=0):
    """The oracle on all host cores on a bounded sample of one scene's default frame: every `stride`-th row at a spp
    sized for ~`seconds` of work. Returns render-only samples/s (b) and, beside it, the time of what src/main.rs:254-256
    brackets as well (a): scene construction before the render and the PNG encode of the full frame after it."""
    import numpy as np
    d = scene_defaults(scene)
    w, h = width or d["width"], height or d["height"]
    O, osc, build_s = oracle_scene(scene)
    threads = O.load().orc_hardware_threads()
    stride = 16 if h >= 400 else 4
    n, rays, dt = cpu_sample(osc, w, h, d["max_depth"], stride, 1, 99, threads)  # calibration (also warms caches)
    spp = max(1, int(seconds * (n / max(dt, 1e-6)) / n))
    n, rays, dt = cpu_sample(osc, w, h, d["max_depth"], stride, spp, 100, threads)
    # the PNG of a full frame (zlib level 6 like the `png` crate's default), timed on a gradient of the same size
    import io
    from PIL import Image
    frame = (np.indices((h, w)).sum(axis=0) % 251).astype(np.uint8)
    t0 = time.perf_counter()
    Image.fromarray(np.stack([frame] * 3 + [np.full_like(frame, 255)], axis=2), "RGBA").save(io.BytesIO(), format="PNG")
    png_s = time.perf_counter() - t0
    rate = n / dt
    full = w * h * d["samples"]
    return {"scene": scene, "name": d["name"], "value": rate, "unit": UNIT, "cores": threads, "kind": "port",
            "rays_per_sample": rays / n,
            "sample": f"every {stride}th row of the {w}x{h} frame ({len(range(stride // 2, h, stride))} rows) x {spp} spp = "
                      f"{n} path samples, {rays} rays, {dt:.2f} s; C++ f64 oracle (the Rust reference cannot be built here)",
            "default_frame": {"path_samples": full, "render_s_extrapolated": full / rate, "scene_build_s": build_s, "png_encode_s": png_s,
                              "build_render_png_s_extrapolated": build_s + full / rate + png_s,
                              "note": "BASELINE.md §3: (a) build + render + PNG as src/main.rs:254-256 times it, (b) render only; "
                                      "the render is linear in spp (src/main.rs:211) and extrapolated from the sample"}}


def cpu_baseline(args):
    """Scene 9 (the headline) with most of the budget, scenes 1, 7 and 8 with a few seconds each."""
    main = cpu_scene_leg(args.scene, args.cpu_seconds, args.width, args.height)
    main["other_scenes"] = [cpu_scene_leg(sc, max(1.0, args.cpu_seconds / 5)) for sc in (1, 7, 8) if sc != args.scene]
    return main


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    d, w, h = workload(args)
    O, osc, _ = oracle_scene(args.scene)
    threads = O.load().orc_hardware_threads()
    stride = 16
    n, rays, dt = cpu_sample(osc, w, h, d["max_depth"], stride, 1, 7, threads)
    # size each step to ~ (90 s / (steps + warmup)), at least 1 spp
    budget = 90.0 / max(1, args.steps + args.warmup)
    spp = max(1, int(budget * (n / max(dt, 1e-6)) / n))
    for i in range(args.warmup):
        cpu_sample(osc, w, h, d["max_depth"], stride, spp, 1000 + i, threads)
    total_n, total_t, total_rays = 0, 0.0, 0
    for i in range(args.steps):
        n, rays, dt = cpu_sample(osc, w, h, d["max_depth"], stride, spp, 2000 + i, threads)
        total_n, total_t, total_rays = total_n + n, total_t + dt, total_rays + rays
    value = total_n / total_t
    sample = (f"each step: every {stride}th row of the {w}x{h} frame x {spp} spp = {n} path samples; "
              f"C++ f64 oracle restating the reference (Rust toolchain absent), {threads} host threads")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total_t / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config(args, d, w, h),
            "details": {"note": "CPU arm: one host process regardless of --gpus"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "rays_per_sec": total_rays / total_t,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ---------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), line.strip()))

    def stop(self, t0=None, t1=None):
        """Rows that arrived inside [t0, t1] (the timed region; a row reports the 200 ms before it). A region
        shorter than the sampling period may hold none: then every row since start() — the warm-up steps run the
        same load — is used and the window says so."""
        if self.proc:
            self.proc.terminate()
        window = "timed region"
        rows = [r for t, r in self.rows if t0 is None or (t0 <= t <= t1 + 0.2)]
        if not rows:
            rows, window = [r for _, r in self.rows], "warm-up + timed region"
        sm, mx, reasons = [], [], set()
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------
def big_scene_leg(R, abi, ctx, n_prims, n_rays, hbm_peak, l2_gbs):
    """The closest-hit kernel outside the cache-resident regime the shipped scenes live in (their flattened form is
    0.5 MB): n_prims random spheres — a BVH + record set several times the 126 MB L2 — built by the device LBVH builder,
    traced by rtx_trace_rays_device with uniformly random rays through the volume (the least coherent case). Reported
    with its own roofline: here HBM bandwidth is a roof that means something."""
    import numpy as np
    import torch
    rng = np.random.default_rng(5)
    side = n_prims ** (1.0 / 3.0) * 3.0
    node_dt = np.dtype([("kind", "<i4"), ("material", "<i4"), ("child", "<i4"), ("n_children", "<i4"), ("f", "<f8", 10)])
    assert node_dt.itemsize == C.sizeof(abi.Node)
    nodes = np.zeros(n_prims + 1, dtype=node_dt)
    nodes["kind"][:n_prims] = abi.NODE_SPHERE
    nodes["child"][:n_prims] = -1
    nodes["f"][:n_prims, :3] = rng.uniform(-side, side, (n_prims, 3))
    nodes["f"][:n_prims, 3] = rng.uniform(0.2, 1.0, n_prims)
    nodes[n_prims] = (abi.NODE_LIST, -1, 0, n_prims, np.zeros(10))
    children = np.arange(n_prims, dtype=np.int32)
    mat, tex = abi.Material(), abi.Texture()
    mat.kind, mat.texture = abi.MAT_LAMBERTIAN, 0
    tex.kind = abi.TEX_SOLID
    tex.f[0] = tex.f[1] = tex.f[2] = 0.5
    desc = abi.SceneDesc()
    desc.nodes = nodes.ctypes.data_as(C.POINTER(abi.Node))
    desc.n_nodes, desc.root = n_prims + 1, n_prims
    desc.children = children.ctypes.data_as(C.POINTER(C.c_int32))
    desc.n_children = n_prims
    desc.materials, desc.n_materials = C.pointer(mat), 1
    desc.textures, desc.n_textures = C.pointer(tex), 1
    cam = desc.camera
    cam.lookfrom[0], cam.lookfrom[1], cam.lookfrom[2] = 0.0, 0.0, -3.0 * side
    cam.view_up[1] = 1.0
    cam.vertical_fov, cam.aspect_ratio, cam.focus_distance, cam.close_time = 40.0, 1.0, 10.0, 1.0
    ctx.set_bvh_builder("lbvh")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sc = R.DeviceScene(ctx, desc)
    torch.cuda.synchronize()
    create_s = time.perf_counter() - t0
    ctx.set_bvh_builder("sah")
    o, tgt = rng.uniform(-side, side, (n_rays, 3)), rng.uniform(-side, side, (n_rays, 3))
    rays = np.zeros(n_rays, dtype=abi.RAY_DTYPE)
    rays["origin"], rays["direction"] = o, tgt - o
    rays["t_min"], rays["t_max"], rays["xi"] = 0.001, np.finfo(np.float64).max, 0.5
    d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1)).cuda()
    d_hits = torch.empty(n_rays * 88, dtype=torch.uint8, device="cuda")
    for _ in range(2):
        sc.trace_device(d_rays, d_hits, n_rays)
    reps = 5
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        sc.trace_device(d_rays, d_hits, n_rays)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    st = sc.trace_stats(d_rays, n_rays)
    info = sc.info()
    hits = d_hits.cpu().numpy().view(abi.HIT_DTYPE)
    # bytes a ray must fetch: 32 per child box tested + 96 per primitive record tested (f64 records), + its own 80 in / 88 out
    a_ray = 32.0 * st["box_tests"] + 96.0 * (st["sphere_tests"] + st["rect_tests"]) + 168.0
    gbs = a_ray * n_rays / (ms * 1e-3) / 1e9
    sc.close()
    return {"primitives": n_prims, "bvh": "device LBVH (Morton codes + radix sort + Karras)", "bvh_nodes": info["bvh_nodes"],
            "scene_bytes": info["device_bytes"], "scene_create_s": create_s, "rays": n_rays, "ms_per_launch": ms,
            "rays_per_sec": n_rays / (ms * 1e-3), "hit_fraction": float(np.mean(hits["prim_id"] >= 0)),
            "per_ray_means": {k: st[k] for k in ("box_tests", "node_visits", "sphere_tests")},
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                         "algorithmic_bytes_per_ray": a_ray, "l2_frac": gbs / l2_gbs,
                         "note": "algorithmic bytes (node pairs 64 B per visit, records 96 B per test, the ray and its hit) against the "
                                 "measured HBM copy bandwidth; the working set is %.0f MB against 126 MB of L2, the rays are incoherent, "
                                 "so a node visit is a dependent, mostly-missing 64-byte fetch: latency, not bandwidth, is what is left "
                                 "between this fraction and 1" % (info["device_bytes"] / 1e6)}}


class Frame:
    """One accumulator + RGBA8 frame of a given size on this rank, with the multi-GPU combine wired up:
      peer  : rank 0's fused reduce + tonemap kernel reads the other accumulators over NVLink (CUDA-IPC mappings)
      slice : every rank reduces + tonemaps 1/N of the pixels and writes them into rank 0's frame (rtx_reduce_tonemap_slice)
      nccl  : rtx_accum_reduce (ncclReduce on the ctx stream, behind the C ABI) + rtx_tonemap_rgba8 on rank 0
    Accumulators are raw cudaMalloc blocks so that they can be exported over CUDA IPC."""

    def __init__(self, env, w, h, combine):
        import torch
        self.env, self.w, self.h = env, w, h
        lib, ctx, abi, dist = env["lib"], env["ctx"], env["abi"], env["dist"]
        rank, world, dev = env["rank"], env["world"], env["dev"]
        self.n_px = w * h
        self.acc_bytes = self.n_px * 16
        self.accum = C.c_void_p()
        abi.check(lib.rtx_malloc(ctx.h, self.acc_bytes, C.byref(self.accum)))
        self.rgba_p = C.c_void_p()
        abi.check(lib.rtx_malloc(ctx.h, self.n_px * 4, C.byref(self.rgba_p)))

        class _Arr:
            __cuda_array_interface__ = {"shape": (h, w, 4), "typestr": "|u1", "data": (self.rgba_p.value, False), "version": 2}
        self.d_rgba = torch.as_tensor(_Arr(), device=dev)

        class _Acc:
            __cuda_array_interface__ = {"shape": (h, w, 4), "typestr": "<f4", "data": (self.accum.value, False), "version": 2}
        self.d_accum = torch.as_tensor(_Acc(), device=dev)
        self.rgba_host = torch.empty((h, w, 4), dtype=torch.uint8).pin_memory()
        self.combine = "local" if world == 1 else combine
        self.all_acc = self.root_rgba = self.peers = self.comm = None
        if world == 1:
            return
        if self.combine == "auto":
            # NCCL behind the C ABI unless the host has no libnccl: measured 30-34 us per 800x800 combine at 2 / 4 / 8 GPUs
            # against 76-169 us (peer) and 84-127 us (slice) with their two host barriers (profiles/r2_combine_ab.json)
            probe = (C.c_uint8 * 128)()
            have = torch.tensor([1.0 if lib.rtx_comm_unique_id(C.byref(probe)) == 0 else 0.0], device=dev)
            dist.all_reduce(have, op=dist.ReduceOp.MIN)
            self.combine = "nccl" if have.item() > 0 else "peer"
        if self.combine in ("peer", "slice"):
            try:
                def export(ptr):
                    hd = (C.c_uint8 * 64)()
                    abi.check(lib.rtx_ipc_export(ctx.h, ptr, C.byref(hd)))
                    return bytes(hd)
                handles = [None] * world
                dist.all_gather_object(handles, (export(self.accum), export(self.rgba_p)))

                def open_(hb):
                    hd = (C.c_uint8 * 64).from_buffer_copy(hb)
                    p = C.c_void_p()
                    abi.check(lib.rtx_ipc_open(ctx.h, C.byref(hd), C.byref(p)))
                    return p.value
                ptrs = [self.accum.value if r == rank else open_(handles[r][0]) for r in range(world)]
                self.all_acc = (C.c_void_p * world)(*ptrs)
                self.peers = (C.c_void_p * (world - 1))(*[ptrs[r] for r in range(world) if r != 0]) if rank == 0 else None
                self.root_rgba = self.rgba_p.value if rank == 0 else open_(handles[0][1])
                ok = torch.ones(1, device=dev)
            except Exception as e:  # noqa: BLE001
                sys.stderr.write(f"[rank {rank}] CUDA IPC unavailable ({e}); combining with NCCL\n")
                ok = torch.zeros(1, device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if ok.item() <= 0:
                self.combine = "nccl"
        if self.combine == "nccl":
            ident = (C.c_uint8 * 128)()
            if rank == 0:
                abi.check(lib.rtx_comm_unique_id(C.byref(ident)))
            box = [bytes(ident)]
            dist.broadcast_object_list(box, src=0)
            ident = (C.c_uint8 * 128).from_buffer_copy(box[0])
            self.comm = C.c_void_p()
            abi.check(lib.rtx_comm_create(ctx.h, world, rank, C.byref(ident), C.byref(self.comm)))

    def zero(self):
        self.env["abi"].check(self.env["lib"].rtx_memset_zero(self.env["ctx"].h, self.accum, self.acc_bytes))

    def render(self, scene_h, spp_begin, spp_count, max_depth, ray_counter=None):
        abi, lib, ctx = self.env["abi"], self.env["lib"], self.env["ctx"]
        p = abi.RenderParams(self.w, self.h, spp_begin, spp_count, max_depth, 0, 1)
        rc = C.c_void_p(ray_counter.data_ptr()) if ray_counter is not None else None
        abi.check(lib.rtx_render(ctx.h, scene_h, C.byref(p), self.accum, rc))

    def combine_and_tonemap(self):
        """every rank's accumulator -> RGBA8 frame on rank 0 (device)."""
        abi, lib, ctx, rank, world = self.env["abi"], self.env["lib"], self.env["ctx"], self.env["rank"], self.env["world"]
        barrier = self.env["barrier"]
        if self.combine == "peer":
            barrier()  # every rank's accumulator is complete
            if rank == 0:
                abi.check(lib.rtx_reduce_tonemap_peers(ctx.h, self.accum, self.peers, world - 1, self.w, self.h, self.rgba_p))
            barrier()  # peers may overwrite their accumulators again
        elif self.combine == "slice":
            barrier()
            abi.check(lib.rtx_reduce_tonemap_slice(ctx.h, self.all_acc, world, rank, self.w, self.h, C.c_void_p(self.root_rgba)))
            barrier()
        elif self.combine == "nccl":
            abi.check(lib.rtx_accum_reduce(ctx.h, self.comm, self.accum, self.w, self.h, 0))
            if rank == 0:
                abi.check(lib.rtx_tonemap_rgba8(ctx.h, self.accum, self.w, self.h, self.rgba_p, 1))
        else:
            abi.check(lib.rtx_reduce_tonemap_peers(ctx.h, self.accum, None, 0, self.w, self.h, self.rgba_p))


def run_ours(args):
    import numpy as np  # noqa: F401
    import torch
    import torch.distributed as dist

    import rttnw_b200 as R
    from rttnw_b200 import abi

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    d, w, h = workload(args)
    assert R.scene_defaults(args.scene) == scene_defaults(args.scene), "bench.py's scene table disagrees with the library's"
    lib = abi.load()
    ctx = R.Context(local)
    desc = R.BuiltinDesc(args.scene)
    scene = R.DeviceScene(ctx, desc)
    info = scene.info()
    dev = torch.device("cuda", local)
    n_px = w * h

    def barrier():
        if world > 1:
            dist.barrier()
    env = {"lib": lib, "ctx": ctx, "abi": abi, "dist": dist, "rank": rank, "world": world, "dev": dev, "barrier": barrier}
    frame = Frame(env, w, h, args.combine)
    combine = frame.combine
    ray_counter = torch.zeros(1, dtype=torch.int64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    step_no = [0]

    def render_step(sc):
        """render spp samples/pixel on this rank, combine on rank 0, tonemap (device RGBA8)."""
        k = step_no[0]
        step_no[0] += 1
        frame.zero()
        frame.render(sc.h, (k * world + rank) * args.spp, args.spp, d["max_depth"], ray_counter)
        frame.combine_and_tonemap()

    def timed(fn, steps, sampler=None, flush_l2=True):
        barrier()
        torch.cuda.synchronize()
        t0 = time.monotonic()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            if flush_l2:
                flush.fill_(1)  # evict L2 between timed steps
            fn()
        ev1.record()
        torch.cuda.synchronize()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), (sampler.stop(t0, time.monotonic()) if sampler else None)

    # ---- device-resident throughput ----
    sampler = ClockSampler(local)  # started ahead of the warm-up: nvidia-smi needs a few hundred ms to deliver its first row
    sampler.start()
    for _ in range(max(3, args.warmup)):
        flush.fill_(1)
        render_step(scene)
    ray_counter.zero_()
    # the render call alone, for the roofline (events on the launching stream, inside the timed region)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    it = iter(kev)

    def step_resident():
        e0, e1 = next(it)
        k = step_no[0]
        step_no[0] += 1
        frame.zero()
        e0.record()
        frame.render(scene.h, (k * world + rank) * args.spp, args.spp, d["max_depth"], ray_counter)
        e1.record()
        frame.combine_and_tonemap()
    ctx.set_profiling(True)  # CUDA events around every 8th shade / trace launch, on the launching stream
    ctx.profile_read(reset=True)
    launches0 = ctx.kernel_launches()
    total_ms, clocks = timed(step_resident, args.steps, sampler)
    launches = ctx.kernel_launches() - launches0
    prof = ctx.profile_read(reset=True)
    ctx.set_profiling(False)
    # the last timed step's outputs, before the legs below reuse the frame's buffers
    outputs = {"accum": frame.d_accum.cpu().numpy(), "frame": frame.d_rgba.cpu().numpy()} if args.dump_outputs and rank == 0 else None
    kern_ms = [a.elapsed_time(b) for a, b in kev]
    rays_rank = int(ray_counter.item())
    samples_total = n_px * args.spp * world * args.steps
    value = samples_total / (total_ms * 1e-3)
    rays_t = torch.tensor([float(rays_rank)], device=dev)
    if world > 1:
        dist.all_reduce(rays_t, op=dist.ReduceOp.SUM)
    rays_total = rays_t.item()

    # ---- end to end through the public API, host buffers ----
    h2d = [0]
    e2e_log = []

    def step_e2e():
        t0 = time.perf_counter()
        sc = R.DeviceScene(ctx, desc)  # flatten + BVH build on the host, H2D of the whole scene
        t1 = time.perf_counter()
        h2d[0] = sc.info()["device_bytes"] + sum(desc.desc.images[i].width * desc.desc.images[i].height * 4
                                                  for i in range(desc.desc.n_images) if desc.desc.images[i].rgba)
        render_step(sc)
        t2 = time.perf_counter()
        if rank == 0:
            frame.rgba_host.copy_(frame.d_rgba, non_blocking=True)  # D2H of the frame
        torch.cuda.current_stream().synchronize()
        t3 = time.perf_counter()
        sc.close()
        t4 = time.perf_counter()
        e2e_log.append((t1 - t0, t2 - t1, t3 - t2, t4 - t3))
    for _ in range(2):
        step_e2e()
    e2e_steps = max(2, min(args.steps, 4))
    e2e_ms, _ = timed(step_e2e, e2e_steps)
    e2e_value = n_px * args.spp * world * e2e_steps / (e2e_ms * 1e-3)
    if rank == 0:
        sys.stderr.write("e2e host phases per step (scene create, render call, sync + D2H, scene destroy) ms: " +
                         "; ".join("/".join(f"{1e3 * x:.1f}" for x in row) for row in e2e_log) + "\n")

    # ---- the frames BASELINE.json's metric names: final scene at 10 000 spp in total (strong scaling), Cornell boxes ----
    frames = {}
    if not args.no_frames:
        def one_frame(number, spp_total, fr, sc):
            dd = scene_defaults(number)
            begin, count = R.shard_spp(spp_total, rank, world)
            rc = torch.zeros(1, dtype=torch.int64, device=dev)

            def go():
                fr.zero()
                chunk = 1 << 12  # (rtx_render takes up to 2^26 spp per call; chunks keep the sample index arithmetic in range)
                for b0 in range(begin, begin + count, chunk):
                    fr.render(sc.h, b0, min(chunk, begin + count - b0), dd["max_depth"], rc)
                fr.combine_and_tonemap()
                if rank == 0:
                    fr.rgba_host.copy_(fr.d_rgba, non_blocking=True)
            ms, _ = timed(go, 1, flush_l2=False)
            rt = torch.tensor([float(rc.item())], device=dev)
            if world > 1:
                dist.all_reduce(rt, op=dist.ReduceOp.SUM)
            n = fr.w * fr.h * spp_total
            return {"scene": number, "name": dd["name"], "width": fr.w, "height": fr.h, "spp_total": spp_total, "spp_per_gpu": count,
                    "seconds": ms * 1e-3, "value": n / (ms * 1e-3), "unit": UNIT, "rays_per_sec": rt.item() / (ms * 1e-3),
                    "scaling": "strong", "timed": "zero + render (this rank's share of the spp) + combine + tonemap + D2H of the frame, "
                    "barrier + synchronize on both sides, max over ranks; run once after the warm-up of the step loop",
                    "reference_default_spp": dd["samples"]}
        if args.scene == 9 and (w, h) == (800, 800):
            frames["final_10k"] = one_frame(9, args.final_spp, frame, scene)
        for name, number in (("cornell_box", 7), ("cornell_smoke", 8)):
            dd = scene_defaults(number)
            sc = R.DeviceScene(ctx, R.BuiltinDesc(number))
            fr = Frame(env, dd["width"], dd["height"], combine if combine != "local" else args.combine)
            fr.zero()
            fr.render(sc.h, 0, 8, dd["max_depth"])  # warm-up: pool allocation for this size, and the first collective of
            fr.combine_and_tonemap()                 # the frame's communicator (NCCL connects lazily: ~1 s)
            ctx.sync()
            frames[name] = one_frame(number, args.cornell_spp, fr, sc)
            sc.close()

    # ---- roofline bookkeeping (rank 0, outside the timed region): counting build of the kernel ----
    line = None
    if rank == 0:
        tmp = scene.new_accum(w, h)
        st = scene.render_counted(tmp, 10_000_000, min(args.spp, 8), seed=1, max_depth=d["max_depth"])
        # SURVEY.md §8d: A_ray = 32 B per child box tested + 32 B per primitive tested + 64 B per instance entered
        a_ray = 32.0 * st["box_tests"] + 32.0 * (st["sphere_tests"] + st["rect_tests"]) + 64.0 * st["instance_enters"]
        f_ray = 12.0 * st["box_tests"] + 30.0 * st["sphere_tests"] + 12.0 * st["rect_tests"] + 40.0 * st["instance_enters"]
        # the dominant kernel is the wavefront trace kernel: every ray of the step goes through exactly one of its
        # launches (one per iteration and pool partition; half of all launches are trace launches). Its launch
        # duration is the mean over the event-bracketed launches (every 8th iteration of partition 0) — measured
        # while the other partition's kernels share the GPU, which is how it runs in production.
        n_it = max(1, prof["iterations"])
        trace_launches = max(1, launches // 2) if prof["iterations"] else args.steps
        kms = prof["trace_ms"] / n_it if prof["iterations"] else sum(kern_ms) / len(kern_ms)  # (megakernel mode: one launch per step)
        rays_per_launch = rays_rank / trace_launches
        algo_gbs = a_ray * rays_per_launch / (kms * 1e-3) / 1e9
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        sms = torch.cuda.get_device_properties(local).multi_processor_count
        counters, why_not = load_counters(args.scene)
        samples_per_s_rank = value / world
        # the roof that does bound the node traffic: L2 read bandwidth, measured on this GPU now (SURVEY.md §8d: l2_gbs)
        l2_gbs = ctx.measure_l2_read()
        hbm = {"algorithmic": {"achieved": algo_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": algo_gbs / hbm_peak,
                               "what": "SURVEY.md §8d algorithmic node + primitive bytes per ray x rays per trace launch / the launch's duration: "
                                       "bytes the traversal must FETCH (from L1/L2: the scene is cache resident), not DRAM traffic"},
               "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s"}
        traffic = None
        if counters:
            dram_per_sample = sum(k["dram_bytes_per_sample"] for k in counters["kernels"].values())
            l2_per_sample = sum(k["l2_bytes_per_sample"] for k in counters["kernels"].values())
            tk = counters["kernels"].get("wf_trace_kernel") or {}
            traffic = tk.get("dram_bytes_per_launch")
            hbm["dram"] = {"achieved": dram_per_sample * samples_per_s_rank / 1e9, "peak": hbm_peak, "unit": "GB/s",
                           "frac": dram_per_sample * samples_per_s_rank / 1e9 / hbm_peak, "bytes_per_sample": dram_per_sample,
                           "what": "dram__bytes_read + dram__bytes_write of every wavefront launch (ncu, per path sample) x this run's samples/s: "
                                   "the ray pool and the accumulator; ncu runs each launch alone and cold, so this is an upper bound"}
            l2 = {"achieved": l2_per_sample * samples_per_s_rank / 1e9, "peak": l2_gbs, "unit": "GB/s",
                  "frac": l2_per_sample * samples_per_s_rank / 1e9 / l2_gbs, "bytes_per_sample": l2_per_sample,
                  "algorithmic_frac": algo_gbs / l2_gbs,
                  "peak_source": "rtx_ctx_measure_l2_read: 16-byte ld.global.cg over a 32 MiB L2-resident buffer, all SMs, this run"}
            issue = issue_roof(counters, samples_per_s_rank, clocks, sms)
            roofline = {"bound": "issue", "achieved": issue["achieved"], "peak": issue["peak"], "unit": issue["unit"], "frac": issue["frac"],
                        "traffic": traffic, "issue": issue, "l2": l2, "hbm": hbm,
                        "counters": {"file": f"profiles/r2_counters_s{args.scene}.json", "kernels_sha": counters["kernels_sha"], "source": counters["source"]}}
        else:
            roofline = {"bound": "issue", "achieved": None, "peak": 4.0 * sms * ((clocks or {}).get("sm_mhz") or 1965.0) * 1e6 / 1e9,
                        "unit": "G warp instructions/s", "frac": None, "traffic": None, "hbm": hbm,
                        "l2": {"peak": l2_gbs, "unit": "GB/s", "algorithmic_frac": algo_gbs / l2_gbs}, "counters": {"unavailable": why_not}}
        roofline.update({
            "kernel": "wf_trace_kernel" if prof["iterations"] else "render_kernel", "kernel_ms_per_launch": kms,
            "launches_per_step": trace_launches / args.steps,
            "kernel_share_of_step": (prof["trace_ms"] if prof["iterations"] else sum(kern_ms)) / total_ms,
            "shade_kernel_share_of_step": prof["shade_ms"] / total_ms, "render_call_ms_per_step": sum(kern_ms) / len(kern_ms),
            "algorithmic_bytes_per_ray": a_ray, "algorithmic_flops_per_ray": f_ray, "rays_per_launch": rays_per_launch,
            "per_ray_means": {k: st[k] for k in ("box_tests", "node_visits", "sphere_tests", "rect_tests", "instance_enters", "medium_tests")},
            "note": "the flattened scene (%.1f MB) and the path pool are L2-resident: what bounds the wavefront is issue slots at the lane "
                    "utilisation divergence leaves (warp_execution_efficiency) and the latency the resident warps cannot cover; HBM and "
                    "L2 bandwidth are far from their roofs (hbm.dram.frac, l2.frac)" % (info["device_bytes"] / 1e6)})
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "dtype_note": "f64 rays, primitive tests, hit points and scatter directions; fp32 BVH boxes (conservative), "
                "textures, throughput and accumulation", "data": "synthetic",
                "config": config(args, d, w, h),
                "details": {"combine": combine, "bvh_nodes": info["bvh_nodes"], "records": info["records"], "scene_bytes": info["device_bytes"],
                            "kernels_sha": kernels_sha()},
                "rays_per_sec": rays_total / (total_ms * 1e-3), "rays_per_sample": rays_total / samples_total,
                "clocks": clocks, "gpu_launches": int(launches),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d[0]), "d2h_bytes_per_step": n_px * 4,
                        "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps},
                "frames": frames,
                "roofline": roofline}
        if world == 1 and args.big_scene > 0:
            try:
                line["big_scene"] = big_scene_leg(R, abi, ctx, args.big_scene, 4_000_000, hbm_peak, l2_gbs)
            except Exception as e:  # noqa: BLE001 (an out-of-memory box must not lose the headline)
                line["big_scene"] = {"unavailable": str(e)}
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit(line)


DUMP_LIMIT = 64 * 10 ** 6  # bytes of .npy data in all


def dump_outputs(out_dir, arrays):
    """Writes each (H, W, C) array as out_dir/<name>.npy in float32. Past DUMP_LIMIT bytes in all, every array keeps the
    same fixed, seeded sample of pixels, whose flat indices go to pixel_index.npy (float64)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    h, w = next(iter(arrays.values())).shape[:2]
    per_px = sum(4 * a.shape[2] for a in arrays.values())
    if h * w * per_px > DUMP_LIMIT:
        k = (DUMP_LIMIT - 4096) // (per_px + 8)  # (room for the index and the .npy headers)
        idx = np.sort(np.random.default_rng(0).choice(h * w, k, replace=False))
        np.save(os.path.join(out_dir, "pixel_index.npy"), idx.astype(np.float64))
        arrays = {name: a.reshape(h * w, -1)[idx] for name, a in arrays.items()}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float32))
    sys.stderr.write(f"outputs of the last timed step: {', '.join(sorted(arrays))} -> {out_dir}\n")


_REAL_STDOUT = None


def claim_stdout():
    """stdout carries exactly one JSON line. Libraries write banners to file descriptor 1 (NCCL prints its version
    there at NCCL_DEBUG >= VERSION): point fd 1 at stderr for the rest of the run and keep the real one for emit()."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    args = parse()
    if args.impl == "reference":
        claim_stdout()
        run_reference(args)
        return
    if args.gpus > 1 and "RANK" not in os.environ:
        # convenience: re-launch under torchrun (the driver launches torchrun itself)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29541", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    claim_stdout()
    run_ours(args)


if __name__ == "__main__":
    main()
