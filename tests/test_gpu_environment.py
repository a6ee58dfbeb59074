"""Environment lighting on the GPU: the miss branch of the render and the feature pass read an HDR lat-long map
(rtx_scene_set_environment; E(d) is written out in include/rttnw_b200.h) instead of the constant background.

Path parity uses the harness of test_gpu_render_paths.py (one path per pixel and call, Philox keyed by (pixel, sample,
bounce)) against orc_render_env (tests/oracle_environment.cpp: the unchanged oracle, the same map, every step of E in
f64). Tolerance of E, derived: the map coordinates are f64 on both sides; the GPU fuses some of their products (the
oracle does not), which moves u and v by a few 2^-53 and E by that times the map's gradient, far below what follows.
The blend is fp32 on the GPU: the fraction fx = (float)(X - x0) is rounded (|error| <= 2^-24, times |b - a| <= 2M),
each difference b - a, product f (b - a) and sum a + f (b - a) is rounded (<= 3 * 2^-24 of a value <= 2M), on two
levels, and the product by the fp32 scale (scale rounded once, product once: 2 * 2^-24). M is the largest texel of
the 2x2 footprint, NOT the result: a lerp between a dark and a bright texel carries the bright one's rounding. So
|E_gpu - E_oracle| <= (2 * (2 + 6) + 2) * 2^-24 * M * scale = 18 * 2^-24 * M * scale, and a path multiplies it by
a throughput <= 1. env_atol takes M = the map's largest texel (the bounded "sun"); the tests add it to the scene
tolerance of test_gpu_render_paths, which covers the rest of the path.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rttnw_b200 as R
from rttnw_b200 import abi
from rttnw_b200 import scene as S
from tests import _oracle as O
from tests._record import record
from tests.test_gpu_adaptive import adaptive, check_prefix, tile_n
from tests.test_gpu_render_paths import MIN_AGREE, RTOL, Z_MAX, compare_paths, gpu_paths, scene_tolerance
from tests.test_host_environment import AXES, expected_colour, oracle_env_lib, sector_map, set_oracle_env

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "rttnw_b200", "lib", "rttnw")
RTX_ERR_INVALID, RTX_ERR_UNSUPPORTED = -1, -5
SCALE = (1.5, 0.8, 1.2)
ROTATION = 37.0


@pytest.fixture(scope="module")
def ctx():
    c = R.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def env_lib(tmp_path_factory):
    return oracle_env_lib(tmp_path_factory)


def sky_map(w=256, h=128, seed=3):
    """A seeded smooth sky with a bright but bounded sun: a Gaussian of peak 40 and a width of ~3 texels."""
    rng = np.random.default_rng(seed)
    v, u = (np.mgrid[0:h, 0:w] + 0.5) / np.array([h, w])[:, None, None]
    ph = rng.random(3) * 2 * np.pi
    img = 0.3 + 0.25 * np.sin(2 * np.pi * u[..., None] * np.array([1, 2, 3]) + ph) * np.sin(np.pi * v[..., None])
    img += (1 - v[..., None]) * np.array([0.2, 0.3, 0.5])
    cu, cv = rng.uniform(0.2, 0.8), rng.uniform(0.2, 0.45)
    sun = 40.0 * np.exp(-(((u - cu) * w) ** 2 + ((v - cv) * h) ** 2) / (2 * 3.0 ** 2))
    img += sun[..., None] * np.array([1.0, 0.9, 0.7])
    return img.astype(np.float32)


def env_atol(img, scale=SCALE):
    return 18 * 2.0 ** -24 * float(img.max()) * max(scale)


class EnvOracle:
    """An oracle scene of the environment library (its own copy of the oracle builds and renders it)."""

    def __init__(self, lib, number=None, desc=None, earth=None):
        self.lib, self._keep = lib, (desc, earth)
        if desc is not None:
            self.h = lib.orc_scene_from_desc(C.byref(desc.desc if hasattr(desc, "desc") else desc), 7)
        else:
            e = None if earth is None else np.ascontiguousarray(earth, dtype=np.uint8)
            self._keep = (None, e)
            self.h = lib.orc_scene_builtin(number, O.SCENE_SEED_BASE + number, None if e is None else e.ctypes.data,
                                           0 if e is None else e.shape[1], 0 if e is None else e.shape[0])
        assert self.h

    def __del__(self):
        try:
            self.lib.orc_scene_free(self.h)
        except Exception:
            pass

    def paths(self, w, h, samples, seed, depth):
        out = []
        for k in range(samples):
            s = np.zeros((h, w, 3))
            self.lib.orc_render_env(self.h, w, h, k, 1, depth, seed, s.ctypes.data, 0)
            out.append(s)
        return np.stack(out)

    def albedo(self, w, h, begin, count, seed):
        al = np.zeros((h, w, 3))
        self.lib.orc_first_vertex_env(self.h, w, h, begin, count, seed, al.ctypes.data, None, None, 0)
        return al


def set_env(lib, sc, img, rotation=0.0, scale=(1.0, 1.0, 1.0)):
    """rtx_scene_set_environment through ctypes, returning the status (for the refusals)."""
    img = np.ascontiguousarray(img, dtype=np.float32)
    env = abi.Environment(img.shape[1], img.shape[0], img.ctypes.data_as(C.POINTER(C.c_float)), rotation,
                          (C.c_double * 3)(*scale))
    return lib.rtx_scene_set_environment(sc.ctx.h, sc.h, C.byref(env))


# ---------------------------------------------------------------------------
# 1. a 1x1 map of float32(background) is the background, bit for bit
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("number", [1, 9])
def test_constant_map_reduces_exactly_to_the_background(ctx, number):
    desc = R.BuiltinDesc(number)
    gsc = R.DeviceScene(ctx, desc)
    plain = gpu_paths(gsc, 64, 64, 4, 31, 50)
    one = np.array(desc.desc.background, dtype=np.float32).reshape(1, 1, 3)
    before = gsc.info()["device_bytes"]
    gsc.set_environment(one, 0.0, 1.0)
    assert gsc.info()["device_bytes"] == before + 2 * 16  # the scale header and one texel
    with_map = gpu_paths(gsc, 64, 64, 4, 31, 50)
    gsc.set_environment(None)
    assert gsc.info()["device_bytes"] == before
    again = gpu_paths(gsc, 64, 64, 4, 31, 50)
    assert with_map.tobytes() == plain.tobytes() and again.tobytes() == plain.tobytes()
    if number == 1:  # a sky scene: the map is what lights it, so a brighter map must change the frame
        gsc.set_environment(one * 2, 0.0, 1.0)
        assert (gpu_paths(gsc, 64, 64, 1, 31, 50) != plain[:1]).any()


def test_first_large_map_is_on_the_device_before_the_next_render(ctx):
    """The first map of a fresh scene, 128 MiB of texels, rendered from at once on the context's stream: the upload
    has finished when set_environment returns, so a constant map of float32(background) gives the background's
    frame bit for bit, and a constant map of another value gives that value in every pixel that sees only the sky."""
    desc = R.BuiltinDesc(2)
    bg = np.array(desc.desc.background, dtype=np.float32)
    plain = gpu_paths(R.DeviceScene(ctx, desc), 64, 64, 1, 17, 50)
    gsc = R.DeviceScene(ctx, desc)
    gsc.set_environment(np.broadcast_to(bg, (2048, 4096, 3)))
    assert gpu_paths(gsc, 64, 64, 1, 17, 50).tobytes() == plain.tobytes()
    cam = S.CameraDescriptor(lookfrom=(0.0, 0.0, 0.0), lookat=(0.0, 0.3, -1.0), vertical_fov=30.0)
    far = S.Sphere((1000.0, 1000.0, 1000.0), 1.0, S.Lambertian((0.5, 0.5, 0.5)))
    sky = R.DeviceScene(ctx, S.Scene(S.List([far]), cam, (0.0, 0.0, 0.0)).to_desc())
    value = np.array([0.25, 1.5, 3.0], dtype=np.float32)
    sky.set_environment(np.broadcast_to(value, (2048, 4096, 3)))
    got = gpu_paths(sky, 64, 64, 1, 17, 1)[0]
    assert (got == value.astype(np.float64)).all()


# ---------------------------------------------------------------------------
# 2. convention: pinhole cameras along the axes see the region the header names
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("rotation", [0.0, 90.0])
def test_cameras_along_the_axes_see_the_named_region(ctx, rotation):
    img, colours = sector_map()
    far = S.Sphere((1000.0, 1000.0, 1000.0), 1.0, S.Lambertian((0.5, 0.5, 0.5)))  # out of every view
    k = 0 if rotation == 0.0 else 1
    for d, keys in AXES.items():
        up = (0.0, 0.0, 1.0) if d[1] != 0 else (0.0, 1.0, 0.0)
        cam = S.CameraDescriptor(lookfrom=(0.0, 0.0, 0.0), lookat=d, view_up=up, vertical_fov=4.0)
        gsc = R.DeviceScene(ctx, S.Scene(S.List([far]), cam, (0.0, 0.0, 0.0)).to_desc())
        gsc.set_environment(img, rotation)
        got = gpu_paths(gsc, 8, 8, 1, 5, 1)[0]
        want = expected_colour(img, colours, keys[k]).astype(np.float64)
        assert (got == want).all(), (rotation, d, got[0, 0], want)
        gsc.close()


# ---------------------------------------------------------------------------
# 3. path parity against the oracle
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("number", [1, 2, 3, 4, 5, 9])
def test_paths_match_the_oracle(ctx, env_lib, number, earth_rgba):
    """64 x 64 pixels x 4 sample indices at depth 50 and at depth 2 under the sky map, rotated and scaled."""
    img = sky_map()
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(number))
    gsc.set_environment(img, ROTATION, SCALE)
    osc = EnvOracle(env_lib, number, earth=earth_rgba)
    set_oracle_env(env_lib, osc.h, img, ROTATION, SCALE)
    rtol, atol = scene_tolerance(number)
    atol += env_atol(img)
    failures = []
    for depth in (2, 50):
        g = gpu_paths(gsc, 64, 64, 4, 41, depth)
        r = osc.paths(64, 64, 4, 41, depth)
        st = compare_paths(g, r, rtol, atol)
        st["min_share_allowed"] = MIN_AGREE[(number, depth)]
        record("environment", f"paths_scene_{number}_depth_{depth}", st)
        print(number, depth, st)
        if st["agree_share"] < st["min_share_allowed"] or max(st["z"]) > Z_MAX:
            failures.append((depth, st))
    assert (r > 0).any(axis=-1).mean() > 0.2  # the map lights a good part of the frame
    assert not failures, failures


# ---------------------------------------------------------------------------
# 4. feature buffers
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("number", [1, 4, 9])
def test_feature_pass_albedo_of_a_miss_is_the_clamped_map(ctx, env_lib, number, earth_rgba):
    """The albedo of every first vertex against orc_first_vertex_env, one sample per call; normals and depth do not
    depend on the map and must equal the feature pass without it."""
    img = sky_map()
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(number))
    osc = EnvOracle(env_lib, number, earth=earth_rgba)
    set_oracle_env(env_lib, osc.h, img, ROTATION, SCALE)
    rtol, atol = scene_tolerance(number)
    bad, total = 0, 0
    for s in range(4):
        plain = gsc.new_aov(64, 64)
        gsc.render_aov(plain, s, 1, seed=23)
        gsc.set_environment(img, ROTATION, SCALE)
        aov = gsc.new_aov(64, 64)
        gsc.render_aov(aov, s, 1, seed=23)
        gsc.set_environment(None)
        ctx.sync()
        g = {k: v.cpu().numpy() for k, v in aov.items()}
        p = {k: v.cpu().numpy() for k, v in plain.items()}
        assert g["normal"].tobytes() == p["normal"].tobytes() and g["depth"].tobytes() == p["depth"].tobytes()
        r = osc.albedo(64, 64, s, 1, 23)
        ok = (np.abs(g["albedo"][..., :3] - r) <= atol + env_atol(img) + rtol * np.abs(r)).all(axis=-1)
        bad += int((~ok).sum())
        total += ok.size
        assert (g["albedo"][..., :3] <= 1).all() and (g["albedo"][..., :3] >= 0).all()
    record("environment", f"aov_scene_{number}", {"pixels": total, "diverging": bad})
    assert bad <= max(1, 1e-4 * total), (bad, total)


# ---------------------------------------------------------------------------
# 5. adaptive sampling keeps its prefix property
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("number", [2, 9])
def test_adaptive_keeps_the_prefix_property(ctx, number):
    img = sky_map()
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(number))
    gsc.set_environment(img, ROTATION, SCALE)
    w, h = 64, 48
    paths = gpu_paths(gsc, w, h, 32, 13, 50)
    acc, aux, stats = adaptive(gsc, 0.02, 8, 8, 32, 13, w=w, h=h)
    n = tile_n(acc)
    assert stats["rounds"] >= 1 and n.min() >= 8 and n.max() <= 32
    check_prefix(acc, aux, paths)


# ---------------------------------------------------------------------------
# 6. refusals
# ---------------------------------------------------------------------------
def test_bad_maps_are_invalid(ctx):
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(2))
    lib = ctx.lib
    good = np.ones((2, 4, 3), dtype=np.float32)
    assert set_env(lib, gsc, good) == 0
    for img, rot, scale in [(np.full((2, 4, 3), np.nan, np.float32), 0.0, (1, 1, 1)),
                            (-good, 0.0, (1, 1, 1)), (good * np.inf, 0.0, (1, 1, 1)),
                            (good, float("inf"), (1, 1, 1)), (good, float("nan"), (1, 1, 1)),
                            (good, 0.0, (1, -1, 1)), (good, 0.0, (1, float("inf"), 1))]:
        assert set_env(lib, gsc, img, rot, scale) == RTX_ERR_INVALID, (rot, scale)
    for w, h in [(0, 2), (2, 0), (-1, 4), (1 << 16, 1 << 15)]:
        env = abi.Environment(w, h, good.ctypes.data_as(C.POINTER(C.c_float)), 0.0, (C.c_double * 3)(1, 1, 1))
        assert lib.rtx_scene_set_environment(ctx.h, gsc.h, C.byref(env)) == RTX_ERR_INVALID, (w, h)
    env = abi.Environment(1, 1, None, 0.0, (C.c_double * 3)(1, 1, 1))
    assert lib.rtx_scene_set_environment(ctx.h, gsc.h, C.byref(env)) == RTX_ERR_INVALID
    assert gsc.info()["device_bytes"] > 9 * 16  # the refusals left the good map in place


@pytest.mark.parametrize("setting", ["RTX_MODE=mega", "RTX_SHADE=1", "RTX_ORDER=1", "counted"])
def test_unsupported_forms_refuse_a_scene_with_a_map(setting, monkeypatch):
    if setting != "counted":
        k, v = setting.split("=")
        monkeypatch.setenv(k, v)
    c = R.Context(0)
    try:
        gsc = R.DeviceScene(c, R.BuiltinDesc(2))
        acc = gsc.new_accum(16, 16)
        p = abi.RenderParams(16, 16, 0, 2, 8, 0, 1)
        st = abi.TraceStats()

        def call():
            if setting == "counted":
                return c.lib.rtx_render_counted(c.h, gsc.h, C.byref(p), acc.data_ptr(), C.byref(st))
            return c.lib.rtx_render(c.h, gsc.h, C.byref(p), acc.data_ptr(), None)

        assert call() == 0  # as before without a map
        gsc.set_environment(sky_map(16, 8))
        assert call() == RTX_ERR_UNSUPPORTED
        abi.check(c.lib.rtx_ctx_set_async(c.h, 1))
        assert call() == RTX_ERR_UNSUPPORTED  # refused at the call, not from a later join
        c.sync()
        if setting != "counted":
            aux = gsc.new_accum(16, 16)
            with pytest.raises(abi.RtxError):
                gsc.render_adaptive(acc, aux, 0.1, 2, 2, 4)
        gsc.set_environment(None)
        assert call() == 0
        c.sync()
        gsc.close()
    finally:
        c.close()


# ---------------------------------------------------------------------------
# 7. ordering against asynchronous renders
# ---------------------------------------------------------------------------
def test_set_environment_is_ordered_between_async_renders(ctx):
    """Queued renders use the map they were queued with: render A (map 1), set map 2, render B, set None, render C."""
    m1, m2 = sky_map(64, 32, 1), sky_map(64, 32, 2)
    w, h = 96, 64
    ref = {}
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(1))
    for key, m in (("a", m1), ("b", m2), ("c", None)):
        gsc.set_environment(m)
        ref[key] = gpu_paths(gsc, w, h, 1, 3, 50)[0]
    c = R.Context(0)
    try:
        abi.check(c.lib.rtx_ctx_set_async(c.h, 1))
        sc = R.DeviceScene(c, R.BuiltinDesc(1))
        acc = {k: sc.new_accum(w, h) for k in ref}
        sc.set_environment(m1)
        sc.render_into(acc["a"], 0, 1, seed=3)
        sc.set_environment(m2)
        sc.render_into(acc["b"], 0, 1, seed=3)
        sc.set_environment(None)
        sc.render_into(acc["c"], 0, 1, seed=3)
        c.sync()
        for k in ref:
            assert acc[k].cpu().numpy()[..., :3].astype(np.float64).tobytes() == ref[k].tobytes(), k
        sc.close()
    finally:
        c.close()


# ---------------------------------------------------------------------------
# 8. front ends: render(env=...) and the CLI
# ---------------------------------------------------------------------------
def test_render_takes_a_path_or_an_array(tmp_path):
    img = sky_map(64, 32)
    R.pfm_write(str(tmp_path / "sky.pfm"), img)
    kw = dict(width=48, height=32, samples=8, seed=5)
    plain = R.render(2, **kw)
    by_path = R.render(2, env=str(tmp_path / "sky.pfm"), env_rotation=30.0, env_scale=2.0, **kw)
    by_array = R.render(2, env=img, env_rotation=30.0, env_scale=(2.0, 2.0, 2.0), **kw)
    assert (np.abs(by_path.astype(int) - by_array.astype(int)) <= 1).all()
    assert (by_path != plain).any()
    for extra in (dict(noise_threshold=0.05), dict(aov_prefix=str(tmp_path / "a")), dict(denoise=True)):
        out = R.render(2, env=img, **kw, **extra)
        assert out.shape == (32, 48, 4)


def cli(args, cwd, timeout=300):
    return subprocess.run([CLI] + args, cwd=cwd, capture_output=True, text=True, timeout=timeout)


def read_png(path):
    return R.png_read_rgba8(str(path)).astype(int)


CLI_PATHS = {"uniform": [], "threaded_checkpoint": ["--checkpoint", "ck"], "adaptive": ["--adaptive", "0.05"],
             "aov": ["--aov", "out"], "denoise": ["--denoise"]}


@pytest.mark.parametrize("path", sorted(CLI_PATHS))
def test_cli_env_on_every_path(tmp_path, path):
    img = sky_map(64, 32)
    R.pfm_write(str(tmp_path / "sky.pfm"), img)
    base = ["2", "--width", "48", "--height", "32", "--spp", "16"] + CLI_PATHS[path]
    r = cli(base + ["--env", "sky.pfm", "--env-rotate", "30", "--env-scale", "2"], tmp_path)
    assert r.returncode == 0, r.stderr
    lit = read_png(tmp_path / "image.png")
    r = cli(base, tmp_path)
    assert r.returncode == 0, r.stderr
    assert (lit != read_png(tmp_path / "image.png")).any()
    if path == "uniform":  # the same frame as render(env=...), up to the fp32 order of the sums
        want = R.render(2, width=48, height=32, samples=16, seed=1, env=img, env_rotation=30.0, env_scale=2.0).astype(int)
        assert (np.abs(lit - want) <= 1).all()
    if path == "threaded_checkpoint":  # resumed with the same --env, the frame is the one rendered in one go
        r = cli(base + ["--env", "sky.pfm", "--env-rotate", "30", "--env-scale", "2", "--chunk", "4", "--stop-after-chunks", "2"], tmp_path)
        assert r.returncode == 3, r.stderr
        r = cli(["2", "--width", "48", "--height", "32", "--spp", "16", "--resume", "ck", "--chunk", "4", "--env", "sky.pfm",
                 "--env-rotate", "30", "--env-scale", "2"], tmp_path)
        assert r.returncode == 0, r.stderr
        assert (np.abs(read_png(tmp_path / "image.png") - lit) <= 1).all()


def test_cli_env_on_two_gpus(tmp_path):
    n = C.c_int()
    abi.check(abi.load().rtx_device_count(C.byref(n)))
    if n.value < 2:
        pytest.skip("needs two devices")
    img = sky_map(64, 32)
    R.pfm_write(str(tmp_path / "sky.pfm"), img)
    r = cli(["2", "--width", "48", "--height", "32", "--spp", "64", "--gpus", "2", "--env", "sky.pfm"], tmp_path)
    assert r.returncode == 0, r.stderr
    want = R.render(2, width=48, height=32, samples=64, seed=1, env=img).astype(int)
    assert (np.abs(read_png(tmp_path / "image.png") - want) <= 1).all()


@pytest.mark.parametrize("args", [["--env", "missing.pfm"], ["--env", "sky.pfm", "--env-rotate", "x"],
                                  ["--env", "sky.pfm", "--env-rotate", "inf"], ["--env", "sky.pfm", "--env-scale", "-1"],
                                  ["--env", "sky.pfm", "--env-scale", "2x"], ["--env-rotate", "10"], ["--env-scale", "2"],
                                  ["--env", "bad.pfm"], ["--env", "sky.png"]])
def test_cli_refuses_bad_env_arguments_before_rendering(tmp_path, args):
    R.pfm_write(str(tmp_path / "sky.pfm"), sky_map(16, 8))
    (tmp_path / "bad.pfm").write_bytes(b"PF\n4 4\n-1\n" + bytes(10))
    R.png_write_rgba8(str(tmp_path / "sky.png"), np.zeros((4, 8, 4), dtype=np.uint8))
    r = cli(["2", "--spp", "4"] + args, tmp_path, timeout=60)
    assert r.returncode == 1 and "--env" in r.stderr, r.stderr
    if args[-1] in ("missing.pfm", "sky.png"):  # no reader ran: the message says what the file is not
        assert "not a readable PFM or Radiance HDR file" in r.stderr, r.stderr
    assert "Scene number" not in r.stdout and not (tmp_path / "image.png").exists()
