"""Python face of the C ABI: `Context`, `DeviceScene`, `render()` — the call a user makes.

Mirrors `fn render(width, aspect, samples, scene)` of src/main.rs:58-233: scene table,
camera, pixel loop, gamma, RGBA8 PNG — with the pixel loop running in the CUDA library.
torch is used for device buffers, streams and torch.distributed only.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

from . import abi

SCENE_SEED_BASE = 0x5254544E57  # "RTTNW"; builtin scene seed = base + scene number (SURVEY.md §8d)
_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_EARTH = os.path.join(_ROOT, "assets", "earth.png")


def png_read_rgba8(path: str) -> np.ndarray:
    lib = abi.load()
    w, h, buf = C.c_int32(), C.c_int32(), C.POINTER(C.c_uint8)()
    abi.check(lib.rtx_png_read_rgba8(path.encode(), C.byref(w), C.byref(h), C.byref(buf)))
    try:
        arr = np.ctypeslib.as_array(buf, shape=(h.value, w.value, 4)).copy()
    finally:
        lib.rtx_buffer_free(buf)
    return arr


def png_write_rgba8(path: str, rgba: np.ndarray) -> None:
    rgba = np.ascontiguousarray(rgba, dtype=np.uint8)
    assert rgba.ndim == 3 and rgba.shape[2] == 4
    abi.check(abi.load().rtx_png_write_rgba8(path.encode(), rgba.shape[1], rgba.shape[0], rgba.ctypes.data))


def scene_defaults(number: int) -> dict:
    """Resolution / spp / depth of the scene table, src/main.rs:66-183,255."""
    d = abi.SceneDefaults()
    abi.check(abi.load().rtx_builtin_scene_defaults(number, C.byref(d)))
    return {"width": d.width, "height": d.height, "samples": d.samples, "max_depth": d.max_depth,
            "name": d.name.decode()}


class BuiltinDesc:
    """One of the nine scenes.rs constructors, as an rtx_scene_desc owned by the library."""

    def __init__(self, number: int, seed: Optional[int] = None, earth_png: Optional[str] = None):
        self.lib = abi.load()
        self.number = number
        self.ptr = C.POINTER(abi.SceneDesc)()
        seed = SCENE_SEED_BASE + number if seed is None else seed
        path = (earth_png or DEFAULT_EARTH).encode()
        abi.check(self.lib.rtx_builtin_scene(number, seed, path, C.byref(self.ptr)))

    @property
    def desc(self) -> abi.SceneDesc:
        return self.ptr.contents

    def __del__(self):
        try:
            if self.ptr:
                self.lib.rtx_scene_desc_free(self.ptr)
        except Exception:
            pass


def flatten_check(desc) -> dict:
    """Host-only: flatten + BVH build + invariants (no GPU)."""
    d = desc.desc if hasattr(desc, "desc") else desc
    a, b, c = C.c_int32(), C.c_int32(), C.c_int32()
    abi.check(abi.load().rtx_flatten_check(C.byref(d), C.byref(a), C.byref(b), C.byref(c)))
    return {"bvh_nodes": a.value, "records": b.value, "prim_ids": c.value}


class Context:
    """One per GPU. Launches on torch's current stream of that device."""

    def __init__(self, device: int = 0):
        import torch
        self.torch = torch
        self.lib = abi.load()
        if not torch.cuda.is_available():
            raise abi.RtxError("no CUDA device: rttnw_b200 has no CPU fallback")
        self.device = device
        torch.cuda.set_device(device)
        self.stream = torch.cuda.current_stream(device)
        self.h = C.c_void_p()
        # torch's default stream has handle 0, which the ABI reads as "create your own": name it explicitly
        # (cudaStreamLegacy == 0x1) so that kernels, torch tensors and torch events share one stream order
        handle = self.stream.cuda_stream or 0x1
        abi.check(self.lib.rtx_ctx_create(device, C.c_void_p(handle), C.byref(self.h)))

    def sync(self) -> None:
        abi.check(self.lib.rtx_ctx_sync(self.h))

    def set_bvh_builder(self, kind: str) -> None:
        """Which builder makes the world BVH of the scenes created from now on: 'sah' (host binned SAH, the
        default), 'lbvh' or 'ploc' (device, faster builds of slower trees), or 'sah_device' (device binned SAH:
        the host builder's policy, trees of host quality)."""
        abi.check(self.lib.rtx_ctx_set_bvh_builder(self.h, {"sah": 0, "lbvh": 1, "ploc": 2, "sah_device": 3}[kind]))

    def set_profiling(self, on: bool) -> None:
        abi.check(self.lib.rtx_ctx_set_profiling(self.h, 1 if on else 0))

    def profile_read(self, reset: bool = True) -> dict:
        a, b, n = C.c_double(), C.c_double(), C.c_uint64()
        abi.check(self.lib.rtx_ctx_profile_read(self.h, C.byref(a), C.byref(b), C.byref(n), 1 if reset else 0))
        return {"shade_ms": a.value, "trace_ms": b.value, "iterations": n.value}

    def measure_l2_read(self, nbytes: int = 0, repeats: int = 0) -> float:
        """GB/s of 16-byte loads over an L2-resident buffer (the bandwidth roof of BVH-node traffic)."""
        g = C.c_double()
        abi.check(self.lib.rtx_ctx_measure_l2_read(self.h, nbytes, repeats, C.byref(g)))
        return g.value

    def kernel_launches(self) -> int:
        n = C.c_uint64()
        abi.check(self.lib.rtx_ctx_kernel_launches(self.h, C.byref(n)))
        return n.value

    def close(self) -> None:
        if self.h:
            self.lib.rtx_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DeviceScene:
    """A flattened scene resident in HBM (rtx_scene)."""

    def __init__(self, ctx: Context, desc):
        self.ctx = ctx
        self.lib = ctx.lib
        self._desc = desc
        d = desc.desc if hasattr(desc, "desc") else desc
        self.h = C.c_void_p()
        abi.check(self.lib.rtx_scene_create(ctx.h, C.byref(d), C.byref(self.h)))

    def info(self) -> dict:
        a, b, c, n = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
        abi.check(self.lib.rtx_scene_info(self.h, C.byref(a), C.byref(b), C.byref(c), C.byref(n)))
        return {"bvh_nodes": a.value, "records": b.value, "xform_ops": c.value, "device_bytes": n.value}

    def close(self) -> None:
        if self.h:
            self.lib.rtx_scene_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- fixed rays (world.hit) ----
    def trace(self, rays: np.ndarray) -> np.ndarray:
        """Host buffers in, host buffers out (H2D + kernel + D2H inside the call)."""
        rays = np.ascontiguousarray(rays)
        assert rays.dtype == np.dtype(abi.RAY_DTYPE)
        hits = np.zeros(rays.shape[0], dtype=abi.HIT_DTYPE)
        abi.check(self.lib.rtx_trace_rays(self.ctx.h, self.h, rays.shape[0], rays.ctypes.data, hits.ctypes.data))
        return hits

    def trace_device(self, d_rays, d_hits, n: int) -> None:
        """torch uint8 tensors holding rtx_ray[n] / rtx_hit[n]; asynchronous."""
        abi.check(self.lib.rtx_trace_rays_device(self.ctx.h, self.h, n, d_rays.data_ptr(), d_hits.data_ptr()))

    def trace_stats(self, d_rays, n: int) -> dict:
        st = abi.TraceStats()
        abi.check(self.lib.rtx_trace_rays_stats(self.ctx.h, self.h, n, d_rays.data_ptr(), C.byref(st)))
        return {k: getattr(st, k) for k, _ in abi.TraceStats._fields_}

    # ---- render ----
    def new_accum(self, width: int, height: int):
        t = self.ctx.torch
        return t.zeros((height, width, 4), dtype=t.float32, device=f"cuda:{self.ctx.device}")

    def render_into(self, accum, spp_begin: int, spp_count: int, seed: int = 1, max_depth: int = 50,
                    ray_counter=None) -> None:
        """Adds `spp_count` samples per pixel (global sample indices spp_begin..) into accum (H, W, 4) fp32."""
        h, w, _ = accum.shape
        assert accum.is_contiguous() and accum.dtype == self.ctx.torch.float32
        p = abi.RenderParams(w, h, spp_begin, spp_count, max_depth, 0, seed)
        rc = ray_counter.data_ptr() if ray_counter is not None else None
        abi.check(self.lib.rtx_render(self.ctx.h, self.h, C.byref(p), accum.data_ptr(), rc))

    def render_counted(self, accum, spp_begin: int, spp_count: int, seed: int = 1, max_depth: int = 50) -> dict:
        """The counting build of the render kernel: total world.hit queries + mean work per query."""
        h, w, _ = accum.shape
        p = abi.RenderParams(w, h, spp_begin, spp_count, max_depth, 0, seed)
        st = abi.TraceStats()
        abi.check(self.lib.rtx_render_counted(self.ctx.h, self.h, C.byref(p), accum.data_ptr(), C.byref(st)))
        return {k: getattr(st, k) for k, _ in abi.TraceStats._fields_}

    def render_adaptive(self, accum, aux, threshold: float, min_spp: int, step_spp: int, max_spp: int, seed: int = 1,
                        max_depth: int = 50, spp_begin: int = 0) -> dict:
        """Adaptive sampling (rtx_render_adaptive): zeroes accum and aux (H, W, 4) fp32, then renders min_spp samples per
        pixel and step_spp more per round to every 8x4 tile whose noise estimate is still >= threshold, up to max_spp.
        Each pixel ends with the samples [spp_begin, spp_begin + n) of the uniform render; aux holds the odd ones.
        Synchronous; returns the stats."""
        h, w, _ = accum.shape
        assert accum.is_contiguous() and aux.is_contiguous() and aux.shape == accum.shape
        p = abi.RenderParams(w, h, spp_begin, max_spp, max_depth, 0, seed)
        ap = abi.AdaptiveParams(threshold, min_spp, step_spp)
        st = abi.AdaptiveStats()
        abi.check(self.lib.rtx_render_adaptive(self.ctx.h, self.h, C.byref(p), C.byref(ap), accum.data_ptr(),
                                               aux.data_ptr(), C.byref(st)))
        return {k: getattr(st, k) for k, _ in abi.AdaptiveStats._fields_}

    def adaptive_error(self, accum, aux):
        """The per-tile error rtx_render_adaptive decides on, for any (accum, aux) pair: (tiles_y, tiles_x) fp32 on the
        device, row 0 = top tiles."""
        h, w, _ = accum.shape
        t = self.ctx.torch
        out = t.empty(((h + 3) // 4, (w + 7) // 8), dtype=t.float32, device=accum.device)
        abi.check(self.lib.rtx_adaptive_error(self.ctx.h, accum.data_ptr(), aux.data_ptr(), w, h, out.data_ptr()))
        return out

    def tonemap(self, accum) -> np.ndarray:
        h, w, _ = accum.shape
        out = np.zeros((h, w, 4), dtype=np.uint8)
        abi.check(self.lib.rtx_tonemap_rgba8(self.ctx.h, accum.data_ptr(), w, h, out.ctypes.data, 0))
        return out


def shard_spp(total_spp: int, rank: int, world_size: int) -> tuple:
    """Samples are i.i.d. (main.rs:211-217): rank r renders global sample indices
    [begin, begin + count) of every pixel. Contiguous, covers [0, total) exactly once."""
    begin = rank * total_spp // world_size
    end = (rank + 1) * total_spp // world_size
    return begin, end - begin


def render(scene_number: int, width: Optional[int] = None, height: Optional[int] = None,
           samples: Optional[int] = None, seed: int = 1, device: int = 0, out_path: Optional[str] = None,
           scene_seed: Optional[int] = None, noise_threshold: Optional[float] = None,
           min_samples: Optional[int] = None) -> np.ndarray:
    """`render(width, aspect, samples, scene)` of src/main.rs:58 on one GPU; returns RGBA8 (H, W, 4)
    and, like the reference, writes it as a PNG when `out_path` is given ("image.png" there).
    With `noise_threshold`, adaptive sampling (DeviceScene.render_adaptive): `samples` is the most a pixel gets,
    `min_samples` the least (default samples / 64, at least 2, even), each later round adds min_samples."""
    d = scene_defaults(scene_number)
    width, height = width or d["width"], height or d["height"]
    samples = samples or d["samples"]
    ctx = Context(device)
    desc = BuiltinDesc(scene_number, scene_seed)
    scene = DeviceScene(ctx, desc)
    accum = scene.new_accum(width, height)
    if noise_threshold is None:
        scene.render_into(accum, 0, samples, seed=seed, max_depth=d["max_depth"])
    else:
        if min_samples is None:
            min_samples = max(2, (samples // 64 + 1) // 2 * 2)
        scene.render_adaptive(accum, scene.new_accum(width, height), noise_threshold, min_samples, min_samples, samples,
                              seed=seed, max_depth=d["max_depth"])
    rgba = scene.tonemap(accum)
    if out_path:
        png_write_rgba8(out_path, rgba)
    scene.close()
    ctx.close()
    return rgba
