"""The device binned-SAH builder (rtx_ctx_set_bvh_builder(ctx, 3), 'sah_device'): the same closest hits as the oracle
and as the host-built tree, trees of host quality, byte-identical rebuilds, and the edge cases of its build rule."""
import numpy as np
import pytest

import rttnw_b200 as R
from rttnw_b200 import abi
from rttnw_b200 import scene as S
from tests import _oracle as O
from tests import _rays as RY
from tests.test_gpu_parity import both, check_rays, gpu_sum, random_tree

pytestmark = pytest.mark.gpu

RTX_ERR_UNSUPPORTED = -5


@pytest.fixture(scope="module")
def ctx():
    c = R.Context(0)
    yield c
    c.close()


def built_with(ctx, kind, desc):
    ctx.set_bvh_builder(kind)
    try:
        return R.DeviceScene(ctx, desc)
    finally:
        ctx.set_bvh_builder("sah")


def random_spheres(n, seed=5):
    rng = np.random.default_rng(seed)
    mat = S.Lambertian((0.5, 0.5, 0.5))
    side = n ** (1 / 3) * 3.0
    items = [S.Sphere(tuple(c), float(r), mat) for c, r in zip(rng.uniform(-side, side, (n, 3)), rng.uniform(0.2, 1.0, n))]
    return S.Scene(S.List(items)).to_desc(), side, rng


def rays_through(side, m, rng):
    o = rng.uniform(-side, side, (m, 3))
    tgt = rng.uniform(-side, side, (m, 3))
    return O.make_rays(o, tgt - o)


def on_device(rays):
    import torch
    return torch.from_numpy(rays.view(np.uint8).reshape(-1)).cuda()


def node_visits(gsc, d_rays, n):
    return gsc.trace_stats(d_rays, n)["node_visits"]


@pytest.mark.parametrize("number", [1, 2, 7, 8, 9])
def test_sah_device_fixed_rays(ctx, number, earth_rgba):
    """Oracle parity of primary and secondary rays, and the same hits as the host-built tree ray for ray (ties aside)."""
    gsc = built_with(ctx, "sah_device", R.BuiltinDesc(number))
    ref_sc = R.DeviceScene(ctx, R.BuiltinDesc(number))
    osc = O.OracleScene.builtin(number, earth=earth_rgba)
    rng = np.random.default_rng(0xB0 + number)
    cam, _ = osc.camera()
    primary = RY.camera_rays(cam, 200000, rng)
    got, ref, st = check_rays(gsc, osc, primary)
    secondary = RY.secondary_rays(ref, primary, rng)
    got2, _, _ = check_rays(gsc, osc, secondary, min_ok=0.95)
    same = ref_sc.trace(secondary)
    agree = (same["prim_id"] == got2["prim_id"]) & np.isclose(same["t"], got2["t"], rtol=1e-12, atol=0)
    assert agree.mean() > 0.95
    assert gsc.info()["bvh_nodes"] >= 1


def test_sah_device_random_trees_and_render(ctx):
    """Moving spheres, rotated and translated boxes, media with general boundaries: oracle parity on twelve random
    trees; then a depth-2 render of scene 9 through the device-built tree against the oracle, same counters."""
    for seed in range(12):
        rng = np.random.default_rng(5000 + seed)
        desc = S.Scene(random_tree(rng)).to_desc()
        ctx.set_bvh_builder("sah_device")
        try:
            gsc, osc = both(ctx, desc, bvh_seed=seed)
        finally:
            ctx.set_bvh_builder("sah")
        n = 30000
        o = rng.uniform(-40, 40, (n, 3))
        target = rng.uniform(-15, 15, (n, 3))
        rays = O.make_rays(o, target - o, time=rng.random(n), xi=rng.random(n) * 0.999 + 0.0005)
        rays["t_min"] = np.where(rng.random(n) < 0.2, -np.inf, 0.001)
        _, ref, _ = check_rays(gsc, osc, rays)
        sec = RY.secondary_rays(ref, rays, rng)
        if sec.shape[0]:
            check_rays(gsc, osc, sec)
    gsc = built_with(ctx, "sah_device", R.BuiltinDesc(9))
    osc = O.OracleScene.builtin(9)
    got = gpu_sum(gsc, 48, 48, 4, seed=3, max_depth=2).cpu().numpy()[..., :3]
    ref, _ = osc.render_sum(48, 48, 4, seed=3, max_depth=2)
    assert np.isclose(got, ref, rtol=2e-3, atol=2e-3).all(axis=2).mean() > 0.97


def test_sah_device_tree_quality(ctx, earth_rgba):
    """Node visits per ray (a deterministic counter of the traversal) on the same rays through each builder's tree:
    the device binned-SAH tree within 5 % of the host SAH tree and below LBVH and PLOC. Measured (node visits over
    those of the host SAH tree): scene 9 camera + secondary rays: sah_device 0.9994, LBVH 1.2705, PLOC 1.0848;
    2e5 random spheres: sah_device 1.0000, LBVH 1.0701, PLOC 1.2328."""
    osc = O.OracleScene.builtin(9, earth=earth_rgba)
    cam, _ = osc.camera()
    rng = np.random.default_rng(0x5A4)
    primary = RY.camera_rays(cam, 200000, rng)
    ref, _ = osc.trace(primary)
    scene9 = np.concatenate([primary, RY.secondary_rays(ref, primary, rng)])
    spheres, side, srng = random_spheres(200_000)
    sphere_rays = rays_through(side, 500_000, srng)
    for desc, rays in ((R.BuiltinDesc(9), scene9), (spheres, sphere_rays)):
        d_rays = on_device(rays)
        visits = {}
        for kind in ("sah", "lbvh", "ploc", "sah_device"):
            gsc = built_with(ctx, kind, desc)
            visits[kind] = node_visits(gsc, d_rays, rays.shape[0])
            gsc.close()
        print({k: round(v / visits["sah"], 4) for k, v in visits.items()})
        assert visits["sah_device"] <= 1.05 * visits["sah"], visits
        assert visits["sah_device"] < visits["lbvh"] and visits["sah_device"] < visits["ploc"], visits


def test_sah_device_builds_are_deterministic(ctx):
    """Node indices come from scans, the float bounds from order-independent min / max: two builds of a scene give
    the same counts, the same traversal counters and the same hits, byte for byte."""
    desc, side, rng = random_spheres(50_000, seed=9)
    rays = rays_through(side, 200_000, rng)
    d_rays = on_device(rays)
    out = []
    for _ in range(2):
        gsc = built_with(ctx, "sah_device", desc)
        out.append((gsc.info(), gsc.trace_stats(d_rays, rays.shape[0]), gsc.trace(rays)))
        gsc.close()
    (ia, sa, ha), (ib, sb, hb) = out
    assert ia == ib and sa == sb
    assert ha.tobytes() == hb.tobytes()


def test_sah_device_large_scene_same_hits_as_host(ctx):
    """2e5 random spheres, 1e6 rays: the same primitive as the host-built tree for every ray that is not an exact tie
    (two primitives at the very same t, where the traversal order decides)."""
    desc, side, rng = random_spheres(200_000, seed=11)
    rays = rays_through(side, 1_000_000, rng)
    host = R.DeviceScene(ctx, desc).trace(rays)
    dev = built_with(ctx, "sah_device", desc).trace(rays)
    same = (host["prim_id"] == dev["prim_id"]) | (host["t"] == dev["t"])
    assert same.all(), int((~same).sum())
    assert (host["prim_id"] >= 0).mean() > 0.3


def test_sah_device_edge_cases(ctx):
    mat = S.Lambertian((0.5, 0.5, 0.5))
    rng = np.random.default_rng(17)

    def parity(desc, n_rays=20000, span=6.0):
        gsc, osc = built_with(ctx, "sah_device", desc), O.OracleScene.from_desc(desc, 7)
        o = rng.uniform(-span, span, (n_rays, 3)) * 3
        t = rng.uniform(-span, span, (n_rays, 3))
        check_rays(gsc, osc, O.make_rays(o, t - o))
        return gsc

    # two items; three at one centre (all centroids coincide, n <= leaf limit: the root holds one leaf)
    two = S.Scene(S.List([S.Sphere((-2, 0, 0), 1.0, mat), S.Sphere((2, 0, 0), 1.0, mat)])).to_desc()
    g = parity(two)
    assert g.info()["bvh_nodes"] == R.DeviceScene(ctx, two).info()["bvh_nodes"]
    three = S.Scene(S.List([S.Sphere((0, 0, 0), r, mat) for r in (0.5, 1.0, 1.5)])).to_desc()
    g = parity(three)
    assert g.info()["bvh_nodes"] == 1 == R.DeviceScene(ctx, three).info()["bvh_nodes"]
    # 1000 concentric spheres (boxes symmetric about 0: one centroid in f64 and in fp32): median splits of the index
    # range, as the host builder makes them
    same = S.Scene(S.List([S.Sphere((0, 0, 0), 0.5 + 0.001 * k, mat) for k in range(1000)])).to_desc()
    g = parity(same)
    assert g.info()["bvh_nodes"] == R.DeviceScene(ctx, same).info()["bvh_nodes"]
    # spheres at 2^k: every plane split cuts off one sphere; deeper than the stack is refused, not built
    clustered = S.Scene(S.List([S.Sphere((2.0 ** k, 0, 0), 0.25, mat) for k in range(80)])).to_desc()
    try:
        gsc = built_with(ctx, "sah_device", clustered)
    except abi.RtxError as e:
        assert f"rtx status {RTX_ERR_UNSUPPORTED}" in str(e)
    else:
        osc = O.OracleScene.from_desc(clustered, 7)
        xs = 2.0 ** rng.integers(0, 80, 4000)
        check_rays(gsc, osc, O.make_rays(np.stack([xs, np.full_like(xs, 5.0), np.zeros_like(xs)], 1), (0, -1, 0)))
    assert ctx.lib.rtx_ctx_set_bvh_builder(ctx.h, 4) == -1
    assert ctx.lib.rtx_ctx_set_bvh_builder(ctx.h, -1) == -1


@pytest.mark.parametrize("form", ["RTX_TRACE=2", "RTX_TRACE=3"])
def test_sah_device_tree_under_other_kernel_forms(form, monkeypatch):
    """Trace forms 2 and 3 stage the first world_node_count nodes of the world BVH in shared memory; the device
    binned-SAH tree has fewer nodes than n - 1 and its top levels first. Same rays, same image as form 1."""
    base = R.Context(0)
    k, v = form.split("=")
    monkeypatch.setenv(k, v)
    other = R.Context(0)
    try:
        out = []
        for c in (base, other):
            c.set_bvh_builder("sah_device")
            gsc = R.DeviceScene(c, R.BuiltinDesc(9))
            acc = gsc.new_accum(160, 120)
            st = gsc.render_counted(acc, 0, 24, seed=11, max_depth=50)
            out.append((acc.cpu().numpy(), st))
            gsc.close()
        (a, sa), (b, sb) = out
        assert sa["rays"] == sb["rays"] and sa["rays"] > 0
        assert (a[..., 3] == 24).all() and (b[..., 3] == 24).all()
        assert np.allclose(a, b, rtol=1e-4, atol=1e-4)
    finally:
        base.close()
        other.close()
