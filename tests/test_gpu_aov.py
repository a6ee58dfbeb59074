"""The feature-buffer pass (rtx_render_aov), path by path against the f64 oracle, and its files.

A call with spp_count = 1 adds exactly one sample per pixel, so each pixel's albedo, normal and distance are those of
the first vertex of ONE path, the path rtx_render follows for (pixel, sample index) with the same seed.
orc_first_vertex (tests/oracle_first_vertex.cpp, compiled on top of the unchanged oracle) follows the same Philox draws
(camera ray, bounce-0 medium flights) through the reference's world.hit and reports, per (pixel, sample), the vertex kind (miss / surface / medium), the material kind and whether
the query made a comparison within 1e-9 of flipping (a grazing tie). Tolerances come from test_gpu_render_paths.py:
RTOL / ATOL for fp32 values of f64 geometry, noise_atol for NoiseTexture values (one evaluation, value itself).

Legitimate divergences, each with a share limit (twice the share the first B200 run measured, floored at 1e-4; that run
found one checker vertex in 73 728 on scene 1 and no other divergence):
  * checker textures: the GPU takes sinf((float)(10 p)), so a point within an ulp of a stripe edge may take the other
    leaf: both albedos are leaves of the scene's checkers, the normal and distance agree;
  * image textures: a fp32 (u, v) may select a texel adjacent to the oracle's (found by tracing the path's camera ray
    through the oracle for the hit's u, v);
  * grazing ties: the oracle flags the query as fragile.
"""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import rttnw_b200 as R
from rttnw_b200 import abi
from rttnw_b200 import scene as S
from tests import _oracle as O
from tests._record import record
from tests.test_gpu_render_paths import (ATOL, CAMERAS, NOISE_SCENES, RTOL, camera_world, material_scene, media_scene,
                                         noise_atol, primary_rays, texel_neighbourhood_codes, to_code)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "rttnw_b200", "lib", "rttnw")
KIND_MISS, KIND_SURFACE, KIND_MEDIUM = 0, 1, 2
FRAGILE = 0x80

# Largest share of (pixel, sample) first vertices of a builtin scene that may diverge, per class (module docstring).
MAX_CHECKER_SHARE = 1e-4
MAX_TEXEL_SHARE = 1e-4
MAX_TIE_SHARE = 1e-4
# Largest share of first vertices another builder's tree may change: ties at the same t are decided by the traversal
# order (the first B200 run measured none on scenes 3, 7, 8, 9 for LBVH, PLOC and the device SAH tree; floor 1e-4).
MAX_BUILDER_SHARE = 1e-4


# ---------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------
SRC = os.path.join(ROOT, "tests", "oracle_first_vertex.cpp")


@pytest.fixture(scope="session")
def fv_lib(tmp_path_factory):
    """tests/oracle_first_vertex.cpp compiled with the oracle's own flags (oracle/Makefile) into a library of its own.
    It carries its own copy of the oracle, so its scenes are built by it too (FirstVertexScene): the world.hit calls of
    a scene read the Philox state of the library that built the scene."""
    mk = open(os.path.join(ROOT, "oracle", "Makefile")).read()
    flags = re.search(r"^CXXFLAGS \?= (.*)$", mk, re.M).group(1).split()
    out = tmp_path_factory.mktemp("oracle_first_vertex") / "liboracle_first_vertex.so"
    subprocess.run([os.environ.get("CXX", "g++"), *flags, "-shared", "-o", str(out), SRC, "-lpthread"], check=True,
                   capture_output=True)
    lib = C.CDLL(str(out))
    sig = {"orc_scene_builtin": (C.c_void_p, [C.c_int, C.c_uint64, C.c_void_p, C.c_int, C.c_int]),
           "orc_scene_from_desc": (C.c_void_p, [C.POINTER(abi.SceneDesc), C.c_uint64]),
           "orc_scene_free": (None, [C.c_void_p]),
           "orc_first_vertex": (C.c_uint64, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_int])}
    for name, (res, args) in sig.items():
        getattr(lib, name).restype, getattr(lib, name).argtypes = res, args
    return lib


class FirstVertexScene:
    """An oracle scene of the first-vertex library (fv_lib)."""

    def __init__(self, lib, number=None, desc=None, earth=None):
        self.lib, self._keep = lib, (desc, earth)
        if desc is not None:
            self.h = lib.orc_scene_from_desc(C.byref(desc.desc if hasattr(desc, "desc") else desc), 7)
        elif earth is not None:
            earth = np.ascontiguousarray(earth, dtype=np.uint8)
            self._keep = (None, earth)
            self.h = lib.orc_scene_builtin(number, O.SCENE_SEED_BASE + number, earth.ctypes.data, earth.shape[1],
                                           earth.shape[0])
        else:
            self.h = lib.orc_scene_builtin(number, O.SCENE_SEED_BASE + number, None, 0, 0)
        assert self.h

    def __del__(self):
        try:
            self.lib.orc_scene_free(self.h)
        except Exception:
            pass

    def sums(self, w, h, begin, count, seed):
        """(albedo (H,W,3), normal (H,W,3), depth (H,W,2), kind (H,W) uint8 or None) sums in float64."""
        al, nm, dp = np.zeros((h, w, 3)), np.zeros((h, w, 3)), np.zeros((h, w, 2))
        kind = np.zeros((h, w), dtype=np.uint8)
        self.lib.orc_first_vertex(self.h, w, h, begin, count, seed, al.ctypes.data, nm.ctypes.data, dp.ctypes.data,
                                  kind.ctypes.data, 0)
        return al, nm, dp, (kind if count == 1 else None)


def gpu_aov(gsc, w, h, begin, count, seed, **kw):
    aov = gsc.new_aov(w, h)
    gsc.render_aov(aov, begin, count, seed=seed, **kw)
    gsc.ctx.sync()
    return {k: v.cpu().numpy() for k, v in aov.items()}


def close(g, r, rtol, atol):
    return (np.abs(g - r) <= atol + rtol * np.abs(r)).all(axis=-1)


def compare_one(g, r, atol_albedo):
    """Per pixel: do albedo, normal and distance agree (and the counts match exactly)?"""
    assert (g["albedo"][..., 3] == 1).all() and (g["normal"][..., 3] == 1).all()
    al = close(g["albedo"][..., :3].astype(np.float64), r[0], RTOL, atol_albedo)
    nm = close(g["normal"][..., :3].astype(np.float64), r[1], RTOL, ATOL)
    dp = close(g["depth"][..., :1].astype(np.float64), r[2][..., :1], RTOL, ATOL) & (g["depth"][..., 1] == r[2][..., 1])
    return al, nm & dp


def checker_leaves(desc):
    """The fp32 colours of the solid leaves of every checker texture of a description."""
    d = desc.desc if hasattr(desc, "desc") else desc
    tex = [d.textures[i] for i in range(d.n_textures)]
    leaves, todo = [], [t for t in tex if t.kind == abi.TEX_CHECKER]
    while todo:
        t = todo.pop()
        for c in (tex[t.a], tex[t.b]):
            if c.kind == abi.TEX_CHECKER:
                todo.append(c)
            elif c.kind == abi.TEX_SOLID:
                leaves.append(np.float32(list(c.f[:3])).astype(np.float64))
    return np.array(leaves).reshape(-1, 3)


@pytest.fixture(scope="module")
def ctx():
    c = R.Context(0)
    yield c
    c.close()


def test_first_vertex_oracle_on_a_known_scene(fv_lib):
    """Without a GPU: a Lambertian sphere, a Metal sphere and a bright light in front of a background outside [0, 1];
    every vertex takes one of the known albedos, surface normals are unit vectors, a miss adds no distance, and the
    medium of a fog ball carries normal 0 and the phase albedo."""
    light = S.XY.rectangle(S.DiffuseLight((3.0, 0.5, 2.0)), (-3, 3), (1.5, 3), 2.0)
    fog = S.ConstantMedium(S.Sphere((0, -2.0, 0), 0.8, S.Dielectric(1.5)), 5.0, (0.2, 0.4, 0.6))
    world = S.List([S.Sphere((-1.2, 0, 0), 1.0, S.Lambertian((0.5, 0.25, 0.75))),
                    S.Sphere((1.2, 0, 0), 1.0, S.Metal((0.9, 0.8, 0.1), 1.0)), light, fog])
    cam = S.CameraDescriptor(lookfrom=(0, 0, -8), lookat=(0, 0, 0), vertical_fov=50.0)
    desc = S.Scene(world, cam, (2.0, 0.5, -1.0)).to_desc()
    al, nm, dp, kind = FirstVertexScene(fv_lib, desc=desc).sums(40, 30, 3, 1, 11)
    vertex, mat = kind & 3, (kind >> 2) & 7
    want = {abi.MAT_LAMBERTIAN: (0.5, 0.25, 0.75), abi.MAT_METAL: (0.9, 0.8, 0.1), abi.MAT_DIFFUSE_LIGHT: (1.0, 0.5, 1.0),
            abi.MAT_ISOTROPIC: (0.2, 0.4, 0.6)}
    for m, rgb in want.items():
        sel = (vertex > 0) & (mat == m)
        assert sel.sum() > 5, m
        assert np.allclose(al[sel], rgb, rtol=0, atol=1e-15), m
    miss = vertex == KIND_MISS
    assert miss.sum() > 50 and np.allclose(al[miss], (1.0, 0.5, 0.0)) and (dp[miss] == 0).all() and (nm[miss] == 0).all()
    surf = vertex == KIND_SURFACE
    assert np.allclose(np.linalg.norm(nm[surf], axis=-1), 1.0) and (dp[surf][:, 1] == 1).all() and (dp[surf][:, 0] > 5).all()
    med = vertex == KIND_MEDIUM
    assert med.sum() > 5 and (mat[med] == abi.MAT_ISOTROPIC).all() and (nm[med] == 0).all()
    al4, _, dp4, k4 = FirstVertexScene(fv_lib, desc=desc).sums(40, 30, 3, 4, 11)
    assert k4 is None and (dp4[..., 1] <= 4).all() and np.isclose(al4[..., 0].max(), 4.0)


# ---------------------------------------------------------------------------
# 1. the nine scenes, path by path
# ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("number", range(1, 10))
def test_builtin_scene_first_vertices(ctx, fv_lib, number, earth_rgba):
    """96 x 96 pixels x 8 sample indices per scene (scene 9 also at 2^31 - 17): every pixel's three buffers agree with
    orc_first_vertex, except the divergences the module docstring allows, each below its share limit."""
    desc = R.BuiltinDesc(number)
    gsc = R.DeviceScene(ctx, desc)
    fvs = FirstVertexScene(fv_lib, number, earth=earth_rgba)
    osc = O.OracleScene.builtin(number, earth=earth_rgba)  # (for the earth texels' (u, v))
    atol_al = noise_atol(NOISE_SCENES[number][0], NOISE_SCENES[number][1]) if number in NOISE_SCENES else ATOL
    leaves = checker_leaves(desc)
    w = h = 96
    begins = list(range(8)) + ([2 ** 31 - 17] if number == 9 else [])
    counts = {"paths": 0, "checker": 0, "texel": 0, "tie": 0, "unexplained": 0}
    for s in begins:
        g = gpu_aov(gsc, w, h, s, 1, 21)
        r = fvs.sums(w, h, s, 1, 21)
        kind = r[3]
        al_ok, geo_ok = compare_one(g, r, atol_al)
        bad = ~(al_ok & geo_ok)
        counts["paths"] += bad.size
        tie = bad & ((kind & FRAGILE) != 0)
        rest = bad & ~tie
        legit = np.zeros_like(rest)
        if rest.any() and leaves.size:  # checker: both albedos are leaves, the geometry agrees
            ga, ra = g["albedo"][..., :3].astype(np.float64), r[0]
            is_leaf = lambda a: (np.abs(a[..., None, :] - leaves) <= 1e-7).all(axis=-1).any(axis=-1)  # noqa: E731
            chk = rest & geo_ok & is_leaf(ga) & is_leaf(ra)
            counts["checker"] += int(chk.sum())
            legit |= chk
        if (rest & ~legit).any() and number == 4 and s < 2 ** 31 - 17:  # earth texels
            idx = np.flatnonzero((rest & ~legit).ravel())
            hits, _ = osc.trace(primary_rays(osc, w, h, 21, idx + s * w * h))
            near = texel_neighbourhood_codes(earth_rgba, hits["u"], hits["v"])
            ga = g["albedo"][..., :3].reshape(-1, 3)[idx].astype(np.float64)
            ok = (hits["prim_id"] >= 0) & geo_ok.ravel()[idx] & (near == to_code(ga)[:, None]).any(axis=1) \
                & (near == to_code(r[0].reshape(-1, 3)[idx])[:, None]).any(axis=1)
            counts["texel"] += int(ok.sum())
            legit.ravel()[idx[ok]] = True
        counts["tie"] += int(tie.sum())
        counts["unexplained"] += int((rest & ~legit).sum())
    shares = {k: counts[k] / counts["paths"] for k in ("checker", "texel", "tie")}
    record("aov", f"scene_{number}", {"counts": counts, "shares": shares})
    print(number, counts)
    assert counts["unexplained"] == 0, counts
    assert shares["checker"] <= MAX_CHECKER_SHARE and shares["texel"] <= MAX_TEXEL_SHARE, counts
    assert shares["tie"] <= MAX_TIE_SHARE, counts


# ---------------------------------------------------------------------------
# 2. materials, camera, media
# ---------------------------------------------------------------------------
def parity(ctx, fv_lib, desc, w, h, samples, seed, atol_albedo=ATOL):
    gsc, osc = R.DeviceScene(ctx, desc), FirstVertexScene(fv_lib, desc=desc)
    out = []
    for s in range(samples):
        g, r = gpu_aov(gsc, w, h, s, 1, seed), osc.sums(w, h, s, 1, seed)
        al_ok, geo_ok = compare_one(g, r, atol_albedo)
        ok = al_ok & geo_ok
        assert ok.all(), (s, np.argwhere(~ok)[:5], r[3][~ok][:5])
        out.append((g, r))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["lambertian", "metal_0", "metal_1.0", "dielectric_outside", "dielectric_inside",
                                  "dielectric_inside_tir", "light_from_behind", "isotropic"])
def test_material_first_vertices(ctx, fv_lib, name):
    """Every material's albedo rule (Metal with fuzz 1 absorbs some scatters and keeps its albedo), glass seen from
    inside (the normal faces the ray), a light of (3, 2, 1) clamped to 1, and the scale-1 noise enclosure."""
    runs = parity(ctx, fv_lib, material_scene(name), 64, 48, 2, 9, noise_atol(1.0, 21.0))
    g, r = runs[0]
    kind = r[3]
    mat = (kind >> 2) & 7
    if name == "light_from_behind":
        light = mat == abi.MAT_DIFFUSE_LIGHT
        solid = light & (g["depth"][..., 0] < 15.0)  # the (3, 2, 1) rectangle, not the noise enclosure
        assert solid.sum() > 50
        assert (g["albedo"][solid][:, :3] == 1.0).all()
    if name.startswith("dielectric"):
        glass = mat == abi.MAT_DIELECTRIC
        assert glass.sum() > 100 and (g["albedo"][glass][:, :3] == 1.0).all()
    if name == "isotropic":
        assert ((kind & 3) == KIND_MEDIUM).sum() > 50


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CAMERAS))
def test_camera_first_vertices(ctx, fv_lib, name):
    """A lens with an off-centre focus, the [0.25, 0.75] shutter over moving spheres, a non-square aspect, and the 1x1,
    7x3 and 33x17 frames (row 0 = top): the distance is measured from the ray's origin on the lens."""
    cam, w, h = CAMERAS[name]
    desc = S.Scene(camera_world(), cam, (0.0, 0.0, 0.0)).to_desc()
    runs = parity(ctx, fv_lib, desc, w, h, 16 if w * h < 64 else 4, 13, noise_atol(4.0, 3.5))
    assert any((r[3] & 3 == KIND_SURFACE).any() for _, r in runs)


@pytest.mark.gpu
@pytest.mark.parametrize("boundary", ["sphere", "cube", "moving_sphere"])
def test_media_first_vertices(ctx, fv_lib, boundary):
    """Media with sphere, rotated-box and moving-sphere boundaries: a medium vertex carries normal 0, the phase
    texture's albedo (0.8, 0.5, 0.3) and the scatter distance (checked against the oracle)."""
    runs = parity(ctx, fv_lib, media_scene(boundary, 40.0), 64, 64, 4, 17)
    n_med = 0
    for g, r in runs:
        med = (r[3] & 3) == KIND_MEDIUM
        n_med += int(med.sum())
        assert (g["normal"][med][:, :3] == 0).all()
        assert np.allclose(g["albedo"][med][:, :3], np.float32([0.8, 0.5, 0.3]), rtol=0, atol=0)
        assert (g["depth"][med][:, 1] == 1).all()
    assert n_med > 100, n_med


# ---------------------------------------------------------------------------
# 3. agreement with the beauty path
# ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("number", [1, 5, 7])
def test_albedo_of_lights_and_misses_is_the_clamped_depth_1_beauty(ctx, fv_lib, number):
    """At max_depth = 1 a sample's radiance is the emission at its first vertex: where the oracle's vertex is a light or
    a miss, the GPU albedo is the GPU beauty clamped to [0, 1] per channel. An rtx_render after an AOV call gives the
    same frame as before it, byte for byte."""
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(number))
    osc = FirstVertexScene(fv_lib, number)
    w, h = 64, 48
    for s in range(2):
        before = gsc.new_accum(w, h)
        gsc.render_into(before, s, 1, seed=5, max_depth=1)
        g = gpu_aov(gsc, w, h, s, 1, 5)
        after = gsc.new_accum(w, h)
        gsc.render_into(after, s, 1, seed=5, max_depth=1)
        ctx.sync()
        b, a = before.cpu().numpy(), after.cpu().numpy()
        assert b.tobytes() == a.tobytes()
        kind = osc.sums(w, h, s, 1, 5)[3]
        sel = (((kind & 3) == KIND_MISS) | (((kind >> 2) & 7) == abi.MAT_DIFFUSE_LIGHT)) & ((kind & FRAGILE) == 0)
        assert sel.sum() > 20
        assert np.array_equal(g["albedo"][sel][:, :3], np.clip(b[sel][:, :3], 0.0, 1.0))


# ---------------------------------------------------------------------------
# 4. determinism, chunking, NULL buffers
# ---------------------------------------------------------------------------
@pytest.mark.gpu
def test_deterministic_chunked_and_null_buffers(ctx):
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(9))
    w, h = 64, 48
    one = gpu_aov(gsc, w, h, 0, 24, 3)
    again = gpu_aov(gsc, w, h, 0, 24, 3)
    for k in one:
        assert one[k].tobytes() == again[k].tobytes(), k
    aov = gsc.new_aov(w, h)
    gsc.render_aov(aov, 0, 8, seed=3)
    gsc.render_aov(aov, 8, 16, seed=3)
    ctx.sync()
    single = [gpu_aov(gsc, w, h, s, 1, 3) for s in range(24)]
    for k in one:
        got = aov[k].cpu().numpy().astype(np.float64)
        bound = 24 * 2.0 ** -24 * sum(np.abs(x[k].astype(np.float64)) for x in single)
        assert (np.abs(got - one[k]) <= bound).all(), k
        assert np.array_equal(got[..., -1], one[k][..., -1])
    assert (one["depth"][..., 1] > 0).mean() > 0.5
    # a buffer passed as NULL is untouched, the others are what the three-buffer call gives
    for keep in ("albedo", "normal", "depth"):
        bufs = gsc.new_aov(w, h)
        for k in bufs:
            if k != keep:
                bufs[k].fill_(7.0)
        gsc.render_aov({keep: bufs[keep]}, 0, 24, seed=3)
        ctx.sync()
        for k in bufs:
            v = bufs[k].cpu().numpy()
            if k == keep:
                assert v.tobytes() == one[k].tobytes()
            else:
                assert (v == 7.0).all()


# ---------------------------------------------------------------------------
# 5. scene and context settings
# ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("setting", ["builder=lbvh", "builder=ploc", "builder=sah_device", "RTX_BVH_WIDE=1", "async"])
def test_settings_do_not_change_the_buffers(ctx, setting, monkeypatch):
    """The same first vertices under every BVH builder (up to exact ties that the traversal order decides), the 4-wide
    BVH setting, and the asynchronous driver (an rtx_render queued before the AOV call)."""
    w, h, spp = 160, 120, 4
    want = {n: gpu_aov(R.DeviceScene(ctx, R.BuiltinDesc(n)), w, h, 0, spp, 23) for n in (3, 7, 8, 9)}
    if "=" in setting and not setting.startswith("builder="):
        k, v = setting.split("=")
        monkeypatch.setenv(k, v)
    c = R.Context(0)
    try:
        if setting.startswith("builder="):
            c.set_bvh_builder(setting.split("=")[1])
        if setting == "async":
            abi.check(c.lib.rtx_ctx_set_async(c.h, 1))
        shares = {}
        for n, ref in want.items():
            gsc = R.DeviceScene(c, R.BuiltinDesc(n))
            if setting == "async":
                acc = gsc.new_accum(w, h)
                gsc.render_into(acc, 0, 8, seed=23)
            got = gpu_aov(gsc, w, h, 0, spp, 23)
            differ = np.zeros((h, w), dtype=bool)
            for k in ref:
                differ |= (got[k] != ref[k]).any(axis=-1)
            shares[n] = float(differ.mean())
            gsc.close()
        record("aov", f"setting_{setting}", shares)
        limit = MAX_BUILDER_SHARE if setting.startswith("builder=") else 0.0
        assert all(v <= limit for v in shares.values()), shares
    finally:
        c.close()


@pytest.mark.gpu
def test_refusals(ctx):
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(7))
    aov = gsc.new_aov(8, 8)
    lib = ctx.lib
    ptrs = [aov[k].data_ptr() for k in ("albedo", "normal", "depth")]

    def call(w=8, h=8, b=0, n=1, d=50, bufs=ptrs):
        p = abi.RenderParams(w, h, b, n, d, 0, 1)
        return lib.rtx_render_aov(ctx.h, gsc.h, C.byref(p), *bufs)

    assert call() == abi.RTX_OK
    assert call(bufs=[None, None, None]) == -1
    for bad in ({"w": 0}, {"h": -1}, {"n": -1}, {"b": -1}, {"n": 2 ** 24 + 1}, {"d": 0}, {"w": 65536, "h": 65536}):
        assert call(**bad) == -1, bad
    with pytest.raises(ValueError):
        gsc.render_aov({"albedo": None}, 0, 1)
    assert call(n=0) == abi.RTX_OK


# ---------------------------------------------------------------------------
# 6. files
# ---------------------------------------------------------------------------
def read_pfm(path):
    with open(path, "rb") as f:
        kind = f.readline().strip()
        w, h = map(int, f.readline().split())
        scale = float(f.readline())
        data = np.frombuffer(f.read(), dtype="<f4")
    c = 3 if kind == b"PF" else 1
    assert kind in (b"PF", b"Pf") and scale == -1.0 and data.size == w * h * c
    img = data.reshape(h, w, c)[::-1]
    return img if c == 3 else img[..., 0]


def test_pfm_round_trip_and_refusals(tmp_path):
    rng = np.random.default_rng(5)
    for shape in ((5, 7, 3), (5, 7), (1, 1), (3, 1, 3)):
        img = rng.normal(size=shape).astype(np.float32)
        p = str(tmp_path / "x.pfm")
        R.pfm_write(p, img)
        assert np.array_equal(read_pfm(p), img)
        head = open(p, "rb").read(2)
        assert head == (b"PF" if img.ndim == 3 else b"Pf")
    lib = abi.load()
    data = np.zeros(64, dtype=np.float32)
    for ch in (0, 2, 4, -1):
        assert lib.rtx_pfm_write(str(tmp_path / "y.pfm").encode(), 2, 2, ch, data.ctypes.data) == -1
    assert lib.rtx_pfm_write(str(tmp_path / "y.pfm").encode(), 0, 2, 3, data.ctypes.data) == -1
    assert lib.rtx_pfm_write(str(tmp_path / "no_dir" / "y.pfm").encode(), 2, 2, 3, data.ctypes.data) == -3
    assert not (tmp_path / "y.pfm").exists()
    with pytest.raises(ValueError):
        R.pfm_write(str(tmp_path / "z.pfm"), np.zeros((2, 2, 4), dtype=np.float32))


@pytest.mark.parametrize("args", [["--aov", "out", "--aov-spp", "0"], ["--aov", "out", "--aov-spp", str(2 ** 24 + 1)],
                                  ["--aov", "out", "--aov-spp", "4x"], ["--aov-spp", "4"]])
def test_cli_refuses_bad_aov_arguments(args, tmp_path):
    r = subprocess.run([CLI, "7", "--spp", "8"] + args, cwd=tmp_path, capture_output=True, text=True, timeout=60)
    assert r.returncode == 1 and "--aov" in r.stderr
    assert "Scene number" not in r.stdout and not list(tmp_path.iterdir())


def check_cli_files(tmp_path, w, h):
    img = R.png_read_rgba8(str(tmp_path / "image.png"))
    beauty = read_pfm(tmp_path / "out.beauty.pfm")
    albedo = read_pfm(tmp_path / "out.albedo.pfm")
    normal = read_pfm(tmp_path / "out.normal.pfm")
    depth = read_pfm(tmp_path / "out.depth.pfm")
    assert beauty.shape == albedo.shape == normal.shape == (h, w, 3) and depth.shape == (h, w)
    code = np.floor(np.clip(np.sqrt(beauty.astype(np.float64)), 0.0, 0.999) * 256.0)
    assert (np.abs(code - img[..., :3]) <= 1).all()
    assert ((albedo >= 0) & (albedo <= 1)).all() and (depth >= 0).all() and (depth > 0).mean() > 0.5
    assert (np.linalg.norm(normal, axis=-1) <= 1.0 + 1e-5).all()
    return beauty


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [[], ["--adaptive", "0.05"], ["--checkpoint", "ck"]])
def test_cli_writes_the_feature_files(extra, tmp_path):
    """The threaded path, the adaptive path and the checkpointing path each write the four PFMs next to image.png."""
    w, h = 64, 48
    r = subprocess.run([CLI, "7", "--width", str(w), "--height", str(h), "--spp", "8", "--aov", "out"] + extra,
                       cwd=tmp_path, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    check_cli_files(tmp_path, w, h)


@pytest.mark.gpu
def test_cli_writes_the_feature_files_with_two_gpus(tmp_path):
    n = C.c_int()
    abi.check(abi.load().rtx_device_count(C.byref(n)))
    if n.value < 2:
        pytest.skip("needs two devices")
    w, h = 64, 48
    r = subprocess.run([CLI, "7", "--width", str(w), "--height", str(h), "--spp", "64", "--gpus", "2", "--aov", "out"],
                       cwd=tmp_path, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    check_cli_files(tmp_path, w, h)


@pytest.mark.gpu
def test_python_render_writes_the_feature_files(tmp_path):
    w, h = 48, 32
    rgba = R.render(7, w, h, 8, out_path=str(tmp_path / "image.png"), aov_prefix=str(tmp_path / "out"), aov_samples=4)
    check_cli_files(tmp_path, w, h)
    assert np.array_equal(rgba, R.png_read_rgba8(str(tmp_path / "image.png")))
