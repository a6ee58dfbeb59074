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
# rtx_denoise's defaults (params == NULL); DESIGN.md §4 gives the reason for each value
DENOISE_DEFAULTS = {"iterations": 5, "sigma_normal": 0.25, "sigma_albedo": 0.1, "sigma_luminance": 8.0}


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


def pfm_write(path: str, image: np.ndarray) -> None:
    """Writes a linear float image (H, W, 3) or (H, W), row 0 = top, as a PFM (rtx_pfm_write)."""
    image = np.ascontiguousarray(image, dtype=np.float32)
    if image.ndim == 2:
        channels = 1
    elif image.ndim == 3 and image.shape[2] == 3:
        channels = 3
    else:
        raise ValueError(f"pfm_write takes (H, W, 3) or (H, W), got {image.shape}")
    abi.check(abi.load().rtx_pfm_write(path.encode(), image.shape[1], image.shape[0], channels, image.ctypes.data))


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

    def denoise(self, accum, half, aov: dict, iterations: int = DENOISE_DEFAULTS["iterations"],
                sigma_normal: float = DENOISE_DEFAULTS["sigma_normal"],
                sigma_albedo: float = DENOISE_DEFAULTS["sigma_albedo"],
                sigma_luminance: float = DENOISE_DEFAULTS["sigma_luminance"]):
        """The feature-guided à-trous filter (rtx_denoise; the exact filter is in include/rttnw_b200.h): accum (H, W, 4)
        as render_into fills it, half (H, W, 4) a value-blind subset of its samples (the aux of render_adaptive, or
        accum cloned after the first half of a uniform render), aov the albedo and normal of DeviceScene.new_aov.
        Returns a new (H, W, 4) fp32 tensor {r, g, b, 1}: a biased, filtered estimate that tonemap() takes as it is.
        Asynchronous on the context's stream; the inputs are not modified."""
        t = self.torch
        h, w, _ = accum.shape
        bufs = (accum, half, aov["albedo"], aov["normal"])
        for b in bufs:
            assert b.is_contiguous() and b.dtype == t.float32 and tuple(b.shape) == (h, w, 4)
        out = t.empty((h, w, 4), dtype=t.float32, device=accum.device)
        p = abi.DenoiseParams(iterations, sigma_normal, sigma_albedo, sigma_luminance)
        abi.check(self.lib.rtx_denoise(self.h, *(b.data_ptr() for b in bufs), w, h, C.byref(p), out.data_ptr()))
        return out

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

    def new_aov(self, width: int, height: int) -> dict:
        """Zeroed feature buffers for render_aov: albedo and normal (H, W, 4) {sum x, sum y, sum z, samples}, depth
        (H, W, 2) {sum distance, samples with a vertex}, fp32 on this context's device."""
        t = self.ctx.torch
        dev = f"cuda:{self.ctx.device}"
        return {"albedo": t.zeros((height, width, 4), dtype=t.float32, device=dev),
                "normal": t.zeros((height, width, 4), dtype=t.float32, device=dev),
                "depth": t.zeros((height, width, 2), dtype=t.float32, device=dev)}

    def render_aov(self, aov: dict, spp_begin: int, spp_count: int, seed: int = 1, max_depth: int = 50) -> None:
        """Adds the first-vertex albedo, normal and distance of the paths (pixel, s), s in [spp_begin, spp_begin +
        spp_count), into the buffers of `aov` (rtx_render_aov; see new_aov). A key that is missing or None is not
        computed. Asynchronous on the context's stream."""
        bufs = [aov.get(k) for k in ("albedo", "normal", "depth")]
        given = [b for b in bufs if b is not None]
        if not given:
            raise ValueError("render_aov needs at least one of albedo, normal, depth")
        h, w = given[0].shape[:2]
        for b, c in zip(bufs, (4, 4, 2)):
            if b is not None:
                assert b.is_contiguous() and b.dtype == self.ctx.torch.float32 and tuple(b.shape) == (h, w, c)
        p = abi.RenderParams(w, h, spp_begin, spp_count, max_depth, 0, seed)
        ptrs = [b.data_ptr() if b is not None else None for b in bufs]
        abi.check(self.lib.rtx_render_aov(self.ctx.h, self.h, C.byref(p), *ptrs))

    def tonemap(self, accum) -> np.ndarray:
        h, w, _ = accum.shape
        out = np.zeros((h, w, 4), dtype=np.uint8)
        abi.check(self.lib.rtx_tonemap_rgba8(self.ctx.h, accum.data_ptr(), w, h, out.ctypes.data, 0))
        return out


def write_aov_files(prefix: str, accum, aov: dict) -> None:
    """PREFIX.beauty.pfm (the linear mean radiance accum.rgb / accum.w the PNG is tonemapped from), PREFIX.albedo.pfm
    and PREFIX.normal.pfm (means over the feature samples; the normals are not renormalised) and PREFIX.depth.pfm (one
    channel: the mean distance over the samples that hit, 0 where none did) — the files the CLI's --aov writes."""
    acc = accum.cpu().numpy().astype(np.float64)
    al, nm, dp = (aov[k].cpu().numpy().astype(np.float64) for k in ("albedo", "normal", "depth"))
    with np.errstate(divide="ignore", invalid="ignore"):
        pfm_write(prefix + ".beauty.pfm", acc[..., :3] / acc[..., 3:4])
        pfm_write(prefix + ".albedo.pfm", al[..., :3] / al[..., 3:4])
        pfm_write(prefix + ".normal.pfm", nm[..., :3] / nm[..., 3:4])
        pfm_write(prefix + ".depth.pfm", np.where(dp[..., 1] > 0, dp[..., 0] / np.maximum(dp[..., 1], 1.0), 0.0))


def shard_spp(total_spp: int, rank: int, world_size: int) -> tuple:
    """Samples are i.i.d. (main.rs:211-217): rank r renders global sample indices
    [begin, begin + count) of every pixel. Contiguous, covers [0, total) exactly once."""
    begin = rank * total_spp // world_size
    end = (rank + 1) * total_spp // world_size
    return begin, end - begin


def render(scene_number: int, width: Optional[int] = None, height: Optional[int] = None,
           samples: Optional[int] = None, seed: int = 1, device: int = 0, out_path: Optional[str] = None,
           scene_seed: Optional[int] = None, noise_threshold: Optional[float] = None,
           min_samples: Optional[int] = None, aov_prefix: Optional[str] = None, aov_samples: int = 16,
           denoise: bool = False) -> np.ndarray:
    """`render(width, aspect, samples, scene)` of src/main.rs:58 on one GPU; returns RGBA8 (H, W, 4)
    and, like the reference, writes it as a PNG when `out_path` is given ("image.png" there).
    With `noise_threshold`, adaptive sampling (DeviceScene.render_adaptive): `samples` is the most a pixel gets,
    `min_samples` the least (default samples / 64, at least 2, even), each later round adds min_samples.
    With `aov_prefix`, also writes the linear frame and the feature buffers of samples [0, aov_samples) as PFMs (see
    write_aov_files): the input of a denoiser such as OIDN or the OptiX denoiser.
    With `denoise`, the returned RGBA (and the PNG) is the tonemap of Context.denoise over the frame, the feature pass
    of samples [0, aov_samples) and a value-blind half of the samples: the adaptive render's odd samples, or a copy of
    the accumulator between the renders of [0, samples / 2) and [samples / 2, samples). With `aov_prefix` as well,
    the denoised frame is also written as PREFIX.denoised.pfm."""
    d = scene_defaults(scene_number)
    width, height = width or d["width"], height or d["height"]
    samples = samples or d["samples"]
    ctx = Context(device)
    desc = BuiltinDesc(scene_number, scene_seed)
    scene = DeviceScene(ctx, desc)
    accum = scene.new_accum(width, height)
    half = None
    if noise_threshold is None:
        if denoise:
            scene.render_into(accum, 0, samples // 2, seed=seed, max_depth=d["max_depth"])
            half = accum.clone()  # (torch's current stream is the context's: ordered between the two renders)
            scene.render_into(accum, samples // 2, samples - samples // 2, seed=seed, max_depth=d["max_depth"])
        else:
            scene.render_into(accum, 0, samples, seed=seed, max_depth=d["max_depth"])
    else:
        if min_samples is None:
            min_samples = max(2, (samples // 64 + 1) // 2 * 2)
        half = scene.new_accum(width, height)
        scene.render_adaptive(accum, half, noise_threshold, min_samples, min_samples, samples,
                              seed=seed, max_depth=d["max_depth"])
    aov = None
    if aov_prefix or denoise:
        aov = scene.new_aov(width, height)
        scene.render_aov(aov, 0, aov_samples, seed=seed, max_depth=d["max_depth"])
    denoised = ctx.denoise(accum, half, aov) if denoise else None
    rgba = scene.tonemap(denoised if denoise else accum)
    if out_path:
        png_write_rgba8(out_path, rgba)
    if aov_prefix:
        write_aov_files(aov_prefix, accum, aov)
        if denoise:
            pfm_write(aov_prefix + ".denoised.pfm", denoised.cpu().numpy()[..., :3])
    scene.close()
    ctx.close()
    return rgba
