"""The render path, one path at a time: every path radiance of the CUDA renderer against the f64 oracle's, and frames
that must not depend on how the work was scheduled compared byte for byte.

Every random draw on both sides is Philox keyed by (pixel, sample, bounce * 256 + purpose, block). A render call with
spp_count = 1 therefore puts exactly one path into each pixel, with one atomicAdd onto 0.0: the accumulator holds that
path's radiance unrounded, and it is the path the oracle's render_sum(spp_begin = s, spp_count = 1) follows. One call
per sample index gives (S, H, W, 3) path radiances to compare element by element.

Tolerances (derived from the fp32 parts of the render path; everything geometric is f64 on both sides):
  * paths that meet no noise texture: throughput, albedo and emission are fp32. Each of at most 50 bounces rounds the
    albedo (2^-24 relative) and one product (2^-24), the radiance sum one more: <= 101 * 2^-24 = 6e-6 relative. The
    test allows rtol = 1e-4, atol = 1e-6.
  * noise textures: NoiseTexture::value is 0.5 (1 + sin(scale z + 10 turb(p))), evaluated in fp32 on (float)p. Rounding
    p moves each coordinate by <= 2^-24 P (P = the largest |coordinate| of a point the texture is evaluated at); octave i
    sees that shift scaled by 2^i and weighted by 2^-i, so with a lattice gradient bound of 5 the seven octaves move the
    sine's argument by <= 10 * 7 * 5 * 2^-24 P, scale z by scale * 2^-24 P, the fp32 products and sums by ~3 * 2^-24
    (scale P + 10): noise_atol(scale, P) = 0.5 * 2^-24 * (350 P + 4 scale P + 30) per unit of emitted radiance the
    value multiplies, counted for two noise hits per path (a third counts as a divergence).
  * checker textures take sinf((float)(10 p)) and image textures a fp32 (u, v): a point within an ulp of a stripe or texel
    edge may take the neighbouring stripe or texel. f64 contraction (nvcc fuses, the oracle is built with
    -ffp-contract=off) moves hit points by ulps, which changes a decision only at an edge or an exact tie. Those paths
    diverge legitimately; each share limit below is twice the share the first B200 run measured, floored.

Every path-parity test also requires the paired bias statistic z = |mean d| / (std d / sqrt n) <= 4 per channel, with
d = gpu - oracle over all paths and differences inside the tolerance set to zero (fp32 albedos are a fixed rounding of
the oracle's f64 values: a consistent 1e-8 bias that is not a bug). One divergent path gives z = 1; k of the same sign
and size give sqrt(k). Seeds are fixed: a given build passes or fails every time.
"""
import ctypes as C
import math

import numpy as np
import pytest

import rttnw_b200 as R
from rttnw_b200 import abi
from rttnw_b200 import scene as S
from tests import _oracle as O
from tests import _rays as RY
from tests._record import record
from tests.test_gpu_parity import both, gpu_sum, random_tree

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-4, 1e-6
Z_MAX = 4.0


@pytest.fixture(scope="module")
def ctx():
    c = R.Context(0)
    yield c
    c.close()


# ---------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------
def gpu_paths(gsc, w, h, samples, seed, depth, begin=0):
    """(S, H, W, 3) float64: the radiance of the one path each pixel gets at sample index begin + s."""
    torch = gsc.ctx.torch
    acc = torch.zeros((samples, h, w, 4), dtype=torch.float32, device=f"cuda:{gsc.ctx.device}")
    for k in range(samples):
        gsc.render_into(acc[k], begin + k, 1, seed=seed, max_depth=depth)
    gsc.ctx.sync()
    a = acc.cpu().numpy()
    assert (a[..., 3] == 1).all()
    return a[..., :3].astype(np.float64)


def oracle_paths(osc, w, h, samples, seed, depth, begin=0):
    return np.stack([osc.render_sum(w, h, 1, seed=seed, spp_begin=begin + k, max_depth=depth)[0] for k in range(samples)])


def compare_paths(g, r, rtol=RTOL, atol=ATOL):
    """Share of paths whose three channels agree within atol + rtol |r|, the largest errors among them, and the
    paired bias statistic z per channel (differences inside the tolerance set to zero)."""
    assert np.isfinite(g).all() and (g >= 0).all()
    d = g - r
    inside = np.abs(d) <= atol + rtol * np.abs(r)
    ok = inside.all(axis=-1)
    dz = np.where(inside, 0.0, d).reshape(-1, 3)
    n = dz.shape[0]
    z = []
    for c in range(3):
        m, sd = dz[:, c].mean(), dz[:, c].std(ddof=1) if n > 1 else 0.0
        z.append(0.0 if m == 0 else (math.inf if sd == 0 else abs(m) / (sd / math.sqrt(n))))
    agree_abs = np.abs(d)[ok]
    agree_rel = (np.abs(d) / np.maximum(np.abs(r), atol))[ok]
    return {"paths": int(ok.size), "agree_share": float(ok.mean()), "diverging": int((~ok).sum()),
            "max_abs_err_agreeing": float(agree_abs.max()) if agree_abs.size else 0.0,
            "max_rel_err_agreeing": float(agree_rel.max()) if agree_rel.size else 0.0,
            "z": [float(v) for v in z], "rtol": rtol, "atol": atol}


def noise_atol(scale, pmax, emission=1.0, hits=1):
    """The module docstring's bound on a path's error from fp32 noise: per evaluation, times the emitted radiance the
    grey value multiplies, times the noise hits allowed per path."""
    return hits * emission * 0.5 * 2.0 ** -24 * (350.0 * pmax + 4.0 * scale * pmax + 30.0)


def check_parity(key, st, min_share):
    st["min_share_allowed"] = min_share
    record("render_paths", key, st)
    print(key, st)
    assert st["agree_share"] >= min_share, (key, st)
    assert max(st["z"]) <= Z_MAX, (key, st)


def per_path(ctx, desc, w, h, samples, seed, depth, begin=0, gsc=None, osc=None):
    gsc = gsc or R.DeviceScene(ctx, desc)
    osc = osc or O.OracleScene.from_desc(desc)
    return gpu_paths(gsc, w, h, samples, seed, depth, begin), oracle_paths(osc, w, h, samples, seed, depth, begin)


# ---------------------------------------------------------------------------
# the nine scenes at every depth the reference uses
# ---------------------------------------------------------------------------
# Noise textures per scene: (largest scale, largest |coordinate| a path can meet a noise texture at, largest radiance the
# value multiplies). Scenes 3 and 5 carry scale-4 noise on the radius-1000 ground sphere centred at O = (0, -1000, 0)
# and on a radius-2 sphere at (0, 2, 0). A point X outside the ground sphere sees only ground points within the tangent
# length sqrt(|X - O|^2 - 1000^2) of itself, and a ray leaving the (convex) ground cannot meet it again, so ground hits
# come from the camera or from the small sphere: scene 3's camera (13, 2, 3) reaches 64.7, the sphere's top (0, 4, 0)
# 89.5, so no coordinate exceeds 92 (P = 100); scene 5's camera (26, 3, 6) reaches 82.0, so P = 26 + 82 -> 110. Scene 3
# sees the sky (1.0), scene 5 a light of 4. Scene 9: the scale-0.1 marble sphere at (220, 280, 300), radius 80, under a
# light of 7 (P = 380).
NOISE_SCENES = {3: (4.0, 100.0, 1.0), 5: (4.0, 110.0, 4.0), 9: (0.1, 380.0, 7.0)}

# Least share of agreeing paths per (scene, depth): 1 - max(twice the diverging share the first B200 run measured, 1e-4).
# Measured (1.5e5 paths each): no diverging path at any depth on scenes 2, 3, 5, 6, 8, 9 and at depth 1 everywhere;
# scene 1 one path at depths 2, 3, 50 (a checker stripe), scene 4 four paths at depths 2, 3, 50 (earth texels), scene 7
# 433 paths (2.9e-3) at depth 50 and none at depths 1-3. The presumed cause, not traced path by path, is exact ties:
# scene 7's later ray generations graze the faces the two boxes share with the floor (MAX_TIES in test_gpu_parity: 1.46 %
# of third-generation rays), the oracle breaks a tie by list order and the GPU by its BVH's traversal order, and the
# LBVH and PLOC trees alone change 0.05-0.09 % of the same scene's depth-50 paths (test_scheduling_does_not_change_a_path).
# Their z is <= 1.4.
MIN_AGREE = {(n, d): 1.0 - 1e-4 for n in range(1, 10) for d in (1, 2, 3, 50)}
MIN_AGREE[(7, 50)] = 1.0 - 5.9e-3


def scene_tolerance(number):
    if number in NOISE_SCENES:
        scale, pmax, emission = NOISE_SCENES[number]
        return RTOL, noise_atol(scale, pmax, emission, hits=2)
    return RTOL, ATOL


@pytest.mark.parametrize("number", range(1, 10))
def test_builtin_scene_paths(ctx, number, earth_rgba):
    """96 x 96 pixels x 16 sample indices (1.5e5 paths) per scene at depths 1, 2, 3 and 50; scene 9 also at one
    sample index just below 2^31, the top of the counter range."""
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(number))
    osc = O.OracleScene.builtin(number, earth=earth_rgba)
    rtol, atol = scene_tolerance(number)
    runs = [(d, 0, 16) for d in (1, 2, 3, 50)]
    if number == 9:
        runs += [(1, 2 ** 31 - 17, 1), (50, 2 ** 31 - 17, 1)]
    failures = []
    for depth, begin, samples in runs:
        g, r = per_path(ctx, None, 96, 96, samples, 21, depth, begin, gsc=gsc, osc=osc)
        st = compare_paths(g, r, rtol, atol)
        key = f"scene_{number}_depth_{depth}" + (f"_begin_{begin}" if begin else "")
        st["min_share_allowed"] = MIN_AGREE[(number, depth)]
        record("render_paths", key, st)
        print(key, st)
        if st["agree_share"] < st["min_share_allowed"] or max(st["z"]) > Z_MAX:
            failures.append((key, st))
    assert not failures, failures


# ---------------------------------------------------------------------------
# textures through emission: at depth 1 the path radiance IS the texture value
# ---------------------------------------------------------------------------
def emitter_scene(tex, shape="sphere", at=(0.0, 0.0, 0.0), size=1.0, lookfrom=None):
    at = np.asarray(at, dtype=np.float64)
    light = S.DiffuseLight(tex)
    if shape == "sphere":
        obj = S.Sphere(tuple(at), size, light)
        lookfrom = lookfrom if lookfrom is not None else tuple(at + np.array([0.3, 0.8, -4.0]) * size)
    elif shape == "rect":
        obj = S.XY.rectangle(light, (at[0] - size, at[0] + size), (at[1] - size, at[1] + size), at[2])
        lookfrom = lookfrom if lookfrom is not None else tuple(at + np.array([0.4, 0.3, -3.0]) * size)
    else:  # the faces of a rotated, translated Cube
        obj = S.Cube((-size, -size, -size), (size, size, size), light).rotate_y(35.0).translate(tuple(at))
        lookfrom = lookfrom if lookfrom is not None else tuple(at + np.array([2.0, 2.5, -4.0]) * size)
    cam = S.CameraDescriptor(lookfrom=lookfrom, lookat=tuple(at), vertical_fov=40.0)
    return S.Scene(S.List([obj]), cam, (0.0, 0.0, 0.0)).to_desc()


CONTINUOUS = {  # name: (texture, centre, radius, noise scale or None)
    "solid": (S.SolidColor((0.3, 0.6, 0.9)), (0, 0, 0), 1.0, None),
    "noise_0.1_origin": (S.NoiseTexture(0.1, seed=11), (0, 0, 0), 2.0, 0.1),
    "noise_4_origin": (S.NoiseTexture(4.0, seed=11), (0, 0, 0), 2.0, 4.0),
    "noise_0.1_negative": (S.NoiseTexture(0.1, seed=12), (-37.3, -12.6, -55.1), 3.0, 0.1),
    "noise_4_negative": (S.NoiseTexture(4.0, seed=12), (-37.3, -12.6, -55.1), 3.0, 4.0),
    "noise_0.1_1e3": (S.NoiseTexture(0.1, seed=13), (1000.5, -999.5, 1000.25), 4.0, 0.1),
    "noise_4_1e3": (S.NoiseTexture(4.0, seed=13), (-1000.5, 999.5, -1000.25), 4.0, 4.0),
}


@pytest.mark.parametrize("name", sorted(CONTINUOUS))
def test_continuous_texture_through_emission(ctx, name):
    """Solid and noise textures have no legitimate divergence: every path within the derived tolerance."""
    tex, at, size, scale = CONTINUOUS[name]
    desc = emitter_scene(tex, "sphere", at, size)
    g, r = per_path(ctx, desc, 64, 64, 4, 5, 1)
    atol = ATOL if scale is None else noise_atol(scale, float(np.abs(np.asarray(at)).max() + size))
    st = compare_paths(g, r, RTOL, atol)
    assert (r > 0).any(axis=-1).mean() > 0.3  # the texture fills a good part of the frame
    check_parity(f"texture_{name}", st, 1.0)


def primary_rays(osc, w, h, seed, idx):
    """The camera rays of the paths at flat indices `idx` of a (S, H, W) gpu_paths / oracle_paths array (spp_begin 0,
    pinhole camera): block (CAMERA, 0) of Philox keyed by the render seed with counter (pixel, sample, 0, 0) holds the
    pixel jitter and the shutter time (main.rs:212-214, camera.rs:63-84)."""
    cam, _ = osc.camera()
    assert cam.aperture == 0.0
    origin, llc, hor, ver, _, _ = RY.camera_basis(cam)
    key = (C.c_uint32 * 2)(seed & 0xFFFFFFFF, seed >> 32)
    s, rest = np.divmod(np.asarray(idx), w * h)
    row, col = np.divmod(rest, w)
    su, sv, tm = (np.zeros(s.shape[0]) for _ in range(3))
    for k in range(s.shape[0]):
        ctr, out = (C.c_uint32 * 4)(int(row[k] * w + col[k]), int(s[k]), 0, 0), (C.c_uint32 * 4)()
        osc.lib.orc_philox4x32_10(C.byref(ctr), C.byref(key), C.byref(out))
        u01 = [(x >> 8) / 16777216.0 for x in out]
        su[k], sv[k], tm[k] = (col[k] + u01[0]) / w, (h - 1 - row[k] + u01[1]) / h, u01[2]
    d = llc + su[:, None] * hor + sv[:, None] * ver - origin
    return O.make_rays(origin, d, time=cam.open_time + (cam.close_time - cam.open_time) * tm)


def to_code(x):
    b = np.rint(np.clip(x, 0, 1) * 255).astype(np.int64)
    return (b[..., 0] << 16) | (b[..., 1] << 8) | b[..., 2]


def texel_neighbourhood_codes(rgba, u, v):
    """Colour codes of the 3 x 3 texels around the one ImageTexture::value (texture.rs:77-106, Q23) picks at (u, v):
    u wraps at the seam, v clamps at the poles. Shape (n, 9)."""
    hgt, wid = rgba.shape[:2]
    i = np.minimum((np.clip(u, 0, 1) * wid).astype(np.int64), wid - 1)
    j = np.minimum(((1 - np.clip(v, 0, 1)) * hgt).astype(np.int64), hgt - 1)
    rgb = rgba[..., :3].astype(np.int64)
    code = (rgb[..., 0] << 16) | (rgb[..., 1] << 8) | rgb[..., 2]
    return np.stack([code[np.clip(j + dj, 0, hgt - 1), (i + di) % wid] for dj in (-1, 0, 1) for di in (-1, 0, 1)], axis=1)


EARTH_CASES = {  # name: (shape, lookfrom relative to the object)
    "sphere_north_pole_and_seam": ("sphere", (-2.2, 3.0, 0.4)),
    "sphere_south_pole_and_seam": ("sphere", (-2.2, -3.0, -0.4)),
    "rectangle": ("rect", None),
    "rotated_cube": ("cube", None),
}
# Largest share of paths that may take a neighbouring texel / stripe: twice the first B200 run's share (measured: none of
# 16384 paths in every case), floored at 1e-4.
MAX_EDGE_SHARE = 1e-4


@pytest.mark.parametrize("name", sorted(EARTH_CASES) + ["checker_nested", "missing_image_cyan"])
def test_discrete_texture_through_emission(ctx, name, earth_rgba):
    """Checker and image textures: every path that differs from the oracle takes the value of a neighbouring stripe
    (one of the checker's leaves) or of a texel adjacent to the one the oracle's hit selects (its camera ray is rebuilt
    from the same Philox draws and traced through the oracle for the hit's (u, v)), and such paths are rare."""
    if name == "checker_nested":
        leaves = [(0.1, 0.2, 0.3), (0.9, 0.8, 0.7), (0.4, 0.9, 0.1), (0.6, 0.05, 0.95)]
        tex = S.CheckerTexture(S.CheckerTexture(leaves[0], leaves[1]), S.CheckerTexture(leaves[2], leaves[3]))
        desc = emitter_scene(tex, "sphere", (0.0, 0.0, 0.0), 1.0)
    elif name == "missing_image_cyan":
        desc = emitter_scene(S.ImageTexture(None), "rect", (0.0, 0.0, 0.0), 1.0)
    else:
        shape, lookfrom = EARTH_CASES[name]
        desc = emitter_scene(S.ImageTexture(earth_rgba), shape, (1.5, -0.5, 2.0), 1.0,
                             None if lookfrom is None else tuple(np.array(lookfrom) + (1.5, -0.5, 2.0)))
    osc = O.OracleScene.from_desc(desc)
    g, r = per_path(ctx, desc, 64, 64, 4, 7, 1, osc=osc)
    st = compare_paths(g, r)
    bad = ~(np.abs(g - r) <= ATOL + RTOL * np.abs(r)).all(axis=-1)
    if name == "checker_nested":
        allowed = np.array(leaves, dtype=np.float32).astype(np.float64)
        legit = (np.abs(g[bad][:, None, :] - allowed[None]) <= 1e-7).all(axis=-1).any(axis=-1)
    elif name == "missing_image_cyan":
        hit = (r > 0).any(axis=-1)
        assert np.array_equal(g[hit], np.broadcast_to([0.0, 1.0, 1.0], g[hit].shape))
        legit = np.zeros(0, dtype=bool)
    else:
        legit = np.zeros(0, dtype=bool)
        if bad.any():
            hits, _ = osc.trace(primary_rays(osc, 64, 64, 7, np.flatnonzero(bad)))
            near = texel_neighbourhood_codes(earth_rgba, hits["u"], hits["v"])
            legit = ((hits["prim_id"] >= 0) & (near == to_code(g[bad])[:, None]).any(axis=1)
                     & (near == to_code(r[bad])[:, None]).any(axis=1))
    st["edge_share"] = float(bad.mean())
    st["max_edge_share_allowed"] = MAX_EDGE_SHARE
    record("render_paths", f"texture_{name}", st)
    print(name, st)
    assert (r > 0).any(axis=-1).mean() > 0.2
    assert legit.all(), (name, g[bad][~legit][:5], r[bad][~legit][:5])
    assert bad.mean() <= MAX_EDGE_SHARE, st
    assert max(st["z"]) <= Z_MAX, st


# ---------------------------------------------------------------------------
# materials at one bounce; the camera; media
# ---------------------------------------------------------------------------
# A scale-1 noise emitter of radius 20 encloses every material scene: what a scattered ray sees depends continuously on
# its direction, so a wrong direction shows in the radiance (a constant background would hide it). A path ends at the
# emitter, so it meets the noise once. Measured: largest error 1.9e-5 against this 2.2e-4; every path agrees.
ENCLOSURE_ATOL = noise_atol(1.0, 21.0)
# Least share of agreeing paths in the feature scenes (materials, media, random trees): all agreed on the first B200 run.
MIN_AGREE_FEATURE = 1.0 - 1e-4


def material_scene(name):
    sky = S.Sphere((0, 0, 0), 20.0, S.DiffuseLight(S.NoiseTexture(1.0, seed=21)))
    cam = S.CameraDescriptor(lookfrom=(0.5, 1.0, -5.0), lookat=(0, 0, 0), vertical_fov=35.0)
    if name == "lambertian":
        obj = [S.Sphere((0, 0, 0), 1.0, S.Lambertian((0.8, 0.4, 0.2)))]
    elif name.startswith("metal_"):
        obj = [S.Sphere((0, 0, 0), 1.0, S.Metal((0.9, 0.7, 0.5), float(name.split("_")[1])))]
    elif name == "dielectric_outside":
        obj = [S.Sphere((0, 0, 0), 1.0, S.Dielectric(1.5))]
    elif name == "dielectric_inside":  # camera rays start inside the glass, 3.2 from the centre of a radius-8 sphere:
        # sin(incidence) <= 3.2 / 8 = 0.4 < 1 / 1.5, so every ray takes the Schlick draw (word 3), none TIR
        obj = [S.Sphere((0, 0, 0), 8.0, S.Dielectric(1.5))]
        cam = S.CameraDescriptor(lookfrom=(0.5, 1.0, -3.0), lookat=(0, 0, 4), vertical_fov=90.0)
    elif name == "dielectric_inside_tir":  # 6.5 from the centre, looking obliquely across: rays that pass more than
        # 8 / 1.5 = 5.33 from the centre meet the glass beyond the critical angle and TIR, the rest take the Schlick draw
        obj = [S.Sphere((0, 0, 0), 8.0, S.Dielectric(1.5))]
        cam = S.CameraDescriptor(lookfrom=(0.0, 0.0, -6.5), lookat=(10.0, 0.0, -0.5), vertical_fov=70.0)
    elif name == "light_from_behind":  # Q24: a DiffuseLight emits on both sides
        obj = [S.XY.rectangle(S.DiffuseLight((3.0, 2.0, 1.0)), (-1, 1), (-1, 1), 1.0),
               S.Sphere((0, 0, 3.0), 1.0, S.Lambertian((0.5, 0.5, 0.5)))]
    else:  # isotropic: a ConstantMedium's phase function
        obj = [S.ConstantMedium(S.Sphere((0, 0, 0), 1.5, S.Dielectric(1.5)), 0.7, (0.3, 0.6, 0.9))]
    return S.Scene(S.List(obj + [sky]), cam, (0.0, 0.0, 0.0)).to_desc()


MATERIALS = ["lambertian", "metal_0", "metal_0.3", "metal_1.0", "dielectric_outside", "dielectric_inside",
             "dielectric_inside_tir", "light_from_behind", "isotropic"]
# Least share of the dielectric_inside_tir camera rays that meet the glass beyond the critical angle, from the camera's
# geometry (computed for the pixel-centre rays of the 64 x 48 frame: 0.59).
MIN_TIR_SHARE = 0.5


def tir_share(osc, w, h):
    """Share of pixel-centre camera rays of a glass sphere of radius 8 at the origin, seen from inside, that meet it
    with 1.5 sin(incidence) > 1; a ray's sin(incidence) is its distance from the centre over the radius."""
    cam, _ = osc.camera()
    origin, llc, hor, ver, _, _ = RY.camera_basis(cam)
    su, sv = np.meshgrid((np.arange(w) + 0.5) / w, (np.arange(h) + 0.5) / h)
    d = llc + su.reshape(-1, 1) * hor + sv.reshape(-1, 1) * ver - origin
    dist = np.linalg.norm(np.cross(origin, d), axis=1) / np.linalg.norm(d, axis=1)
    return float((1.5 * dist / 8.0 > 1.0).mean())


@pytest.mark.parametrize("name", MATERIALS)
def test_material_paths(ctx, name):
    """Every scatter() at depth 2 (one bounce, then the emitter) and depth 3. Metal with fuzz 1 absorbs some rays."""
    desc = material_scene(name)
    gsc, osc = both(ctx, desc)
    for depth in (2, 3):
        g, r = per_path(ctx, desc, 64, 48, 4, 9, depth, gsc=gsc, osc=osc)
        st = compare_paths(g, r, RTOL, ENCLOSURE_ATOL)
        if name == "dielectric_inside_tir":
            # a reflected ray stays inside the sphere, meets the glass again and ends at depth 2 or 3 with nothing: the
            # oracle's paths are black at least as often as the camera rays are beyond the critical angle
            st["tir_share_of_camera_rays"] = tir_share(osc, 64, 48)
            st["oracle_black_share"] = float((r == 0).all(axis=-1).mean())
            assert st["tir_share_of_camera_rays"] >= MIN_TIR_SHARE, st
            assert st["oracle_black_share"] >= st["tir_share_of_camera_rays"] - 0.02, st
        check_parity(f"material_{name}_depth_{depth}", st, MIN_AGREE_FEATURE)


def camera_world():
    tex = S.NoiseTexture(4.0, seed=31)
    light = S.DiffuseLight(tex)
    return S.List([S.Sphere((0, 0, 0), 1.0, light), S.Sphere((-2.5, 0.3, 2.0), 1.0, light),
                   S.Sphere((2.0, -0.5, -2.0), 0.7, light),
                   S.MovingSphere(((0, 1.8, 0), (0.8, 2.2, 0)), (0, 1), 0.5, light),
                   S.MovingSphere(((1.5, 1.0, 1.0), (1.5, -1.0, 1.0)), (0.2, 0.9), 0.6, light)])


CAMERAS = {  # name: (camera, width, height)
    "lens_off_centre_focus": (S.CameraDescriptor(lookfrom=(1, 1, -8), lookat=(0, 0, 0), vertical_fov=40.0,
                                                 aperture=1.2, focus_distance=5.3), 64, 64),
    "shutter_0.25_0.75": (S.CameraDescriptor(lookfrom=(0, 1, -8), lookat=(0, 0.5, 0), vertical_fov=40.0,
                                             open_time=0.25, close_time=0.75), 64, 64),
    "aspect_2.35": (S.CameraDescriptor(lookfrom=(0, 1, -8), lookat=(0, 0, 0), vertical_fov=30.0, aspect_ratio=2.35), 94, 40),
    "frame_1x1": (S.CameraDescriptor(lookfrom=(0, 0, -8), lookat=(0, 0, 0), vertical_fov=10.0), 1, 1),
    "frame_7x3": (S.CameraDescriptor(lookfrom=(0, 1, -8), lookat=(0, 0, 0), vertical_fov=30.0, aspect_ratio=7 / 3), 7, 3),
    "frame_33x17": (S.CameraDescriptor(lookfrom=(0, 1, -8), lookat=(0, 0, 0), vertical_fov=30.0, aspect_ratio=33 / 17), 33, 17),
}


@pytest.mark.parametrize("name", sorted(CAMERAS))
def test_camera_paths(ctx, name):
    """Camera::ray with a lens, a shutter interval other than [0, 1] over moving spheres, a non-square aspect and
    ragged frames (row 0 is the top row). The emitters carry a scale-4 noise near the origin, so a pixel's value is a
    continuous function of where its ray meets them."""
    cam, w, h = CAMERAS[name]
    desc = S.Scene(camera_world(), cam, (0.0, 0.0, 0.0)).to_desc()
    g, r = per_path(ctx, desc, w, h, 16 if w * h < 64 else 4, 13, 1)
    assert (r > 0).any()
    check_parity(f"camera_{name}", compare_paths(g, r, RTOL, noise_atol(4.0, 3.5)), 1.0)


def media_scene(boundary, focus):
    wall = S.XY.rectangle(S.Lambertian((0.7, 0.6, 0.5)), (-10, 10), (-10, 10), 6.0)
    floor = S.XZ.rectangle(S.Lambertian((0.4, 0.5, 0.4)), (-10, 10), (-10, 10), -4.0)
    light = S.XZ.rectangle(S.DiffuseLight((6.0, 6.0, 6.0)), (-3, 3), (-3, 3), 7.0)
    if boundary == "sphere":
        b = S.Sphere((0, 0, 0), 3.0, S.Dielectric(1.5))
    elif boundary == "cube":
        b = S.Cube((-2, -2, -2), (2, 2, 2), S.Lambertian((0.5, 0.5, 0.5))).rotate_y(30.0).translate((0.5, 0.0, 0.5))
    else:
        b = S.MovingSphere(((-1, 0, 0), (1, 0.5, 0)), (0, 1), 2.5, S.Lambertian((0.5, 0.5, 0.5)))
    # mean free path 1 / 0.15 = 6.7: about the distance from the medium to the wall behind it
    med = S.ConstantMedium(b, 0.15, (0.8, 0.5, 0.3))
    cam = S.CameraDescriptor(lookfrom=(0, 1, -12), lookat=(0, 0, 0), vertical_fov=40.0, focus_distance=focus)
    return S.Scene(S.List([wall, floor, light, med]), cam, (0.3, 0.4, 0.5)).to_desc()


@pytest.mark.parametrize("boundary", ["sphere", "cube", "moving_sphere"])
@pytest.mark.parametrize("focus", [40.0, 0.05])
def test_media_paths(ctx, boundary, focus, monkeypatch):
    """media_after (the render path's free-flight filter) against the oracle at depth 50, and byte for byte against
    RTX_SHADE=1, whose media_prepass takes the other route to the same answer. Camera directions have length ~focus:
    media_after scales the segment by an upper bound of |d|, and a wrong bound would skip a test it must run."""
    desc = media_scene(boundary, focus)
    gsc = R.DeviceScene(ctx, desc)
    g, r = per_path(ctx, desc, 64, 64, 4, 17, 50, gsc=gsc)
    check_parity(f"media_{boundary}_focus_{focus}", compare_paths(g, r), MIN_AGREE_FEATURE)
    monkeypatch.setenv("RTX_SHADE", "1")
    other = R.Context(0)
    try:
        g1 = gpu_paths(R.DeviceScene(other, desc), 64, 64, 4, 17, 50)
    finally:
        other.close()
    assert g1.tobytes() == g.tobytes()


def test_random_tree_paths(ctx):
    """The twelve random trees of test_gpu_parity (every material and hittable, media with general boundaries) seen
    by a camera looking into the tree: per-path parity at depth 50."""
    cam = S.CameraDescriptor(lookfrom=(5, 12, -60), lookat=(0, 0, 0), vertical_fov=45.0)
    failures = []
    for seed in range(12):
        rng = np.random.default_rng(1000 + seed)
        desc = S.Scene(random_tree(rng), cam, (0.6, 0.7, 0.8)).to_desc()
        gsc, osc = both(ctx, desc, bvh_seed=seed)
        g, r = per_path(ctx, desc, 48, 48, 4, 19, 50, gsc=gsc, osc=osc)
        st = compare_paths(g, r)
        st["min_share_allowed"] = MIN_AGREE_FEATURE
        record("render_paths", f"random_tree_{seed}", st)
        print(seed, st)
        if st["agree_share"] < MIN_AGREE_FEATURE or max(st["z"]) > Z_MAX:
            failures.append((seed, st))
    assert not failures, failures


# ---------------------------------------------------------------------------
# bit-exact invariance at spp = 1
# ---------------------------------------------------------------------------
INVARIANT_SCENES = (3, 7, 8, 9)
INV_W, INV_H, INV_S = 160, 120, 4


def frames(c, number, builder=None):
    if builder:
        c.set_bvh_builder(builder)
    gsc = R.DeviceScene(c, R.BuiltinDesc(number))
    try:
        return gpu_paths(gsc, INV_W, INV_H, INV_S, 23, 50)
    finally:
        gsc.close()


@pytest.fixture(scope="module")
def default_frames():
    c = R.Context(0)
    try:
        yield {n: frames(c, n) for n in INVARIANT_SCENES}
    finally:
        c.close()


DRIVER = ["RTX_WF_SLOTS=1152", "RTX_WF_SLOTS=2048 RTX_WF_STREAMS=3", "RTX_WF_STREAMS=1", "RTX_WF_STREAMS=4",
          "RTX_WF_BATCH=1", "async", "RTX_ORDER=1"]
FORMS = ["RTX_TRACE=2", "RTX_TRACE=3", "RTX_TRACE=4", "RTX_SHADE=1", "RTX_PERLIN_SMEM=0", "RTX_BVH_WIDE=1", "RTX_MODE=mega"]
BUILDERS = ["builder=lbvh", "builder=ploc", "builder=sah_device"]


# Largest share of depth-50 paths another builder's tree may change, per scene: twice the share the first B200 run
# measured, floored at 1e-4 (measured: scene 7 LBVH 8.85e-4, PLOC 4.82e-4; every other scene and the device SAH tree 0).
BUILDER_MAX_SHARE = {"lbvh": {7: 1.8e-3}, "ploc": {7: 9.7e-4}, "sah_device": {}}


@pytest.mark.parametrize("setting", DRIVER + FORMS + BUILDERS)
def test_scheduling_does_not_change_a_path(setting, default_frames, monkeypatch):
    """At spp = 1 a pixel's value does not depend on scheduling, summation order or pool layout. The driver settings
    (pool size, partitions, refills, batching, the asynchronous driver, ray ordering) touch no ray arithmetic, and the
    kernel forms (trace forms 2-4, the first shade form, the global-memory Perlin table, the 4-wide BVH, the megakernel)
    find the same closest hit in the same tree: all must give the default build's frames byte for byte (measured: they
    do). A tree from another builder gives the same closest hit except where two primitives tie at the very same t and
    the traversal order picks the winner, so a small share of long paths may differ (BUILDER_MAX_SHARE)."""
    builder = None
    if setting.startswith("builder="):
        builder = setting.split("=")[1]
    elif setting != "async":
        for kv in setting.split():
            k, v = kv.split("=")
            monkeypatch.setenv(k, v)
    limit = {n: BUILDER_MAX_SHARE[builder].get(n, 1e-4) if builder else 0.0 for n in INVARIANT_SCENES}
    c = R.Context(0)
    try:
        if setting == "async":
            abi.check(c.lib.rtx_ctx_set_async(c.h, 1))
        result = {}
        for n in INVARIANT_SCENES:
            got = frames(c, n, builder)
            differ = (got != default_frames[n]).any(axis=-1)
            result[n] = float(differ.mean())
        record("render_paths", f"bit_exact_{setting.replace(' ', '_')}",
               {"differing_path_share": {f"scene_{n}": v for n, v in result.items()},
                "max_share_allowed": {f"scene_{n}": limit[n] for n in INVARIANT_SCENES}})
        assert all(result[n] <= limit[n] for n in INVARIANT_SCENES), (result, limit)
    finally:
        c.close()


def test_chunked_call_is_the_sum_of_single_paths(ctx):
    """One call with spp_count = 4 equals the sum of the four spp = 1 frames, within the bound on fp32 summation
    order (4 * 2^-24 * sum |x| per pixel)."""
    for n in (7, 9):
        gsc = R.DeviceScene(ctx, R.BuiltinDesc(n))
        single = gpu_paths(gsc, 96, 72, 4, 29, 50)
        acc = gpu_sum(gsc, 96, 72, 4, seed=29).cpu().numpy().astype(np.float64)
        assert (acc[..., 3] == 4).all()
        bound = 4 * 2.0 ** -24 * np.abs(single).sum(axis=0)
        assert (np.abs(acc[..., :3] - single.sum(axis=0)) <= bound).all()
        assert (single.sum(axis=0) > 0).any(axis=-1).mean() > 0.1


# ---------------------------------------------------------------------------
# tonemap edges: rtx_tonemap_rgba8, rtx_reduce_tonemap_peers (no peers), rtx_reduce_tonemap_slice (one rank)
# ---------------------------------------------------------------------------
def tonemap_reference(acc):
    """main.rs:217-225 in float64 on the fp32 sums: mean, sqrt, clamp(0, 0.999) (NaN stays NaN), * 256, `as u8`
    (truncation, NaN -> 0, saturating)."""
    s, n = acc[:, :3].astype(np.float64), acc[:, 3:4].astype(np.float64)
    with np.errstate(all="ignore"):
        x = np.sqrt(s / n)
        x = np.where(np.isnan(x), np.nan, np.clip(x, 0.0, 0.999)) * 256.0
        t = 256.0 * np.sqrt(s / n)
        near = np.isfinite(t) & (np.abs(t - np.rint(t)) <= 2.0 ** -21 * np.maximum(t, 1.0)) & (t > 0.5) & (t < 256.5)
    q = np.where(np.isnan(x), 0.0, np.floor(x)).astype(np.uint8)
    return q, near


def tonemap_inputs():
    f = np.float32
    rows = []
    for n in (1.0, 2.0, 3.0, 7.0, 100.0, 12345.0, 2.0 ** 24):
        for k in range(256):
            b = f((k / 256.0) ** 2 * n)
            rows.append([b, np.nextafter(b, f(np.inf)), np.nextafter(b, f(-np.inf)), n])
            up2 = np.nextafter(np.nextafter(b, f(np.inf)), f(np.inf))
            dn2 = np.nextafter(np.nextafter(b, f(-np.inf)), f(-np.inf))
            rows.append([up2, dn2, f(0.9990001 ** 2 * n * (1 + k / 64.0)), n])  # ... and values above 0.999^2
    special = [0.0, -0.0, -1.0, -1e-30, np.nan, np.inf, -np.inf, 1e30, 3e38]
    for cnt in (0.0, 1.0, 2.0, 2.0 ** 24):
        for a in special:
            for b in special:
                rows.append([a, b, 0.5, cnt])
    acc = np.array(rows, dtype=np.float32)
    pad = (-acc.shape[0]) % 64
    acc = np.concatenate([acc, np.tile(np.array([[0.25, 0.5, 0.75, 1.0]], dtype=np.float32), (pad, 1))])
    assert acc.shape[0] >= 1024
    return acc


def test_tonemap_edges(ctx):
    import torch
    acc = tonemap_inputs()
    w = 64
    h = acc.shape[0] // w
    d_acc = torch.from_numpy(acc.reshape(h, w, 4)).cuda()
    lib = ctx.lib
    one = np.zeros((h, w, 4), dtype=np.uint8)
    abi.check(lib.rtx_tonemap_rgba8(ctx.h, d_acc.data_ptr(), w, h, one.ctypes.data, 0))
    peers_out = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda")
    d_copy = d_acc.clone()
    abi.check(lib.rtx_reduce_tonemap_peers(ctx.h, d_copy.data_ptr(), None, 0, w, h, peers_out.data_ptr()))
    slice_out = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda")
    ptrs = (C.c_void_p * 1)(d_acc.data_ptr())
    abi.check(lib.rtx_reduce_tonemap_slice(ctx.h, ptrs, 1, 0, w, h, slice_out.data_ptr()))
    ctx.sync()
    assert np.array_equal(peers_out.cpu().numpy(), one) and np.array_equal(slice_out.cpu().numpy(), one)
    assert d_copy.cpu().numpy().tobytes() == acc.reshape(h, w, 4).tobytes()  # no peers: the sum is the input
    got = one.reshape(-1, 4)
    assert (got[:, 3] == 255).all()
    ref, near = tonemap_reference(acc)
    diff = got[:, :3].astype(int) - ref.astype(int)
    exact_off = (diff != 0) & ~near
    assert not exact_off.any(), (acc[exact_off.any(axis=1)][:5], got[exact_off.any(axis=1)][:5], ref[exact_off.any(axis=1)][:5])
    assert (np.abs(diff) <= 1).all()
    with np.errstate(all="ignore"):
        nan_like = np.isnan(acc[:, :3]) | (acc[:, :3] < 0) | ((acc[:, :3] == 0) & (acc[:, 3:4] == 0))
    assert (got[:, :3][nan_like] == 0).all()
    record("render_paths", "tonemap_edges", {"pixels": int(acc.shape[0]), "near_boundary": int(near.sum()),
                                             "off_by_one_near_boundary": int((diff != 0).sum())})
