"""Host-side logic that needs no GPU: the C-ABI library loads and exports every declared symbol,
scene flattening + BVH invariants, the builtin scenes agree with the oracle's restatement of
scenes.rs, PNG I/O, spp sharding (incl. a world_size-2 gloo run). No compute entry point is
called here (there is no CPU compute path to call)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import rttnw_b200 as R
from rttnw_b200 import abi
from rttnw_b200 import scene as S
from tests import _oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    lib = abi.load()
    header = open(os.path.join(ROOT, "include", "rttnw_b200.h")).read()
    declared = set(re.findall(r"\b(rtx_[a-z0-9_]+)\s*\(", header))
    declared -= {"rtx_status"}
    assert len(declared) >= 30
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
        assert name in abi.SIGNATURES, f"{name} has no ctypes signature"
    assert lib.rtx_abi_version() == 1


def test_rust_bindings_declare_the_same_symbols():
    """rust/rttnw-b200-sys cannot be compiled here (no Rust toolchain): at least keep its extern block and the
    header in step, name by name."""
    header = open(os.path.join(ROOT, "include", "rttnw_b200.h")).read()
    declared = set(re.findall(r"\b(rtx_[a-z0-9_]+)\s*\(", header)) - {"rtx_status"}
    ffi = open(os.path.join(ROOT, "rust", "rttnw-b200-sys", "src", "ffi.rs")).read()
    bound = set(re.findall(r"pub fn (rtx_[a-z0-9_]+)", ffi))
    assert bound == declared, (declared - bound, bound - declared)


def test_struct_sizes_match_header():
    # the sizes written next to the typedefs in include/rttnw_b200.h
    assert C.sizeof(abi.Node) == 96 and C.sizeof(abi.Material) == 40 and C.sizeof(abi.Texture) == 48
    assert C.sizeof(abi.Ray) == 80 and C.sizeof(abi.Hit) == 88
    assert C.sizeof(abi.Perlin) == 256 * 3 * 8 + 3 * 256 * 4


def test_compute_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    lib = abi.load()
    h = C.c_void_p()
    assert lib.rtx_ctx_create(0, None, C.byref(h)) == -2  # RTX_ERR_CUDA, not a CPU fallback
    assert b"cuda" in lib.rtx_last_error().lower()
    with pytest.raises(abi.RtxError):
        R.Context(0)


def test_scene_table_matches_main_rs():  # src/main.rs:66-183,255
    expect = {1: (400, 225, 100), 2: (400, 225, 100), 3: (400, 225, 100), 4: (400, 225, 100), 5: (400, 225, 400),
              6: (600, 600, 200), 7: (600, 600, 200), 8: (600, 600, 200), 9: (800, 800, 10000)}
    for n, (w, h, s) in expect.items():
        d = R.scene_defaults(n)
        assert (d["width"], d["height"], d["samples"], d["max_depth"]) == (w, h, s, 50)
    assert R.scene_defaults(9)["name"] == "final_scene"
    with pytest.raises(abi.RtxError, match="There is no scene 10"):
        R.scene_defaults(10)
    with pytest.raises(abi.RtxError):
        R.BuiltinDesc(0)


def test_builtin_scenes_flatten_and_match_oracle_inventory(earth_rgba):
    for n in range(1, 10):
        desc = R.BuiltinDesc(n)
        info = R.flatten_check(desc)
        osc = O.OracleScene.builtin(n, earth=earth_rgba)
        assert info["prim_ids"] == osc.prim_count, f"scene {n}"
        cam, bg = osc.camera()
        assert bytes(cam) == bytes(desc.desc.camera)
        assert tuple(desc.desc.background) == bg
    # final scene: 2400 ground rectangles + 1000 instanced spheres + loose primitives
    info = R.flatten_check(R.BuiltinDesc(9))
    assert info["records"] >= 3400 and info["bvh_nodes"] < 2 * info["records"]


def test_builtin_scene_is_seeded():
    a, b, c = R.BuiltinDesc(1, seed=5), R.BuiltinDesc(1, seed=5), R.BuiltinDesc(1, seed=6)

    def nodes(d):
        return bytes((abi.Node * d.desc.n_nodes).from_address(C.addressof(d.desc.nodes.contents)))
    assert nodes(a) == nodes(b) and nodes(a) != nodes(c)


def test_perlin_tables_of_builtin_scene_match_oracle():
    # scene 3 draws only the Perlin tables: same SplitMix64 stream on both sides
    desc = R.BuiltinDesc(3, seed=1234)
    tab = abi.Perlin()
    O.load().orc_perlin_generate(1234, C.byref(tab))
    assert bytes(desc.desc.perlins[0]) == bytes(tab)


def test_flatten_rejects_malformed_descriptions():
    mat = S.Lambertian((0.5, 0.5, 0.5))
    d = S.Scene(S.List([S.Sphere((0, 0, 0), 1.0, mat)])).to_desc()
    d.desc.nodes[0].material = 7
    with pytest.raises(abi.RtxError, match="material"):
        R.flatten_check(d)
    d = S.Scene(S.List([S.Sphere((0, 0, 0), 1.0, mat)])).to_desc()
    d.desc.root = 99
    with pytest.raises(abi.RtxError, match="root"):
        R.flatten_check(d)
    inner = S.ConstantMedium(S.Sphere((0, 0, 0), 1.0, mat), 0.1, (1, 1, 1))
    d = S.Scene(S.List([S.ConstantMedium(inner, 0.1, (1, 1, 1))])).to_desc()
    with pytest.raises(abi.RtxError, match="ConstantMedium"):
        R.flatten_check(d)


def test_flatten_invariants_on_random_trees():
    rng = np.random.default_rng(11)
    mat = S.Lambertian((0.5, 0.5, 0.5))
    for trial in range(6):
        items = []
        for _ in range(int(rng.integers(1, 60))):
            kind = rng.integers(0, 5)
            c = tuple(rng.uniform(-50, 50, 3))
            if kind == 0:
                items.append(S.Sphere(c, float(rng.uniform(0.1, 5)), mat))
            elif kind == 1:
                items.append(S.MovingSphere((c, tuple(np.array(c) + rng.uniform(-2, 2, 3))), (0, 1), 1.0, mat))
            elif kind == 2:
                plane = [S.XY, S.XZ, S.YZ][int(rng.integers(0, 3))]
                a, b = sorted(rng.uniform(-30, 30, 2)), sorted(rng.uniform(-30, 30, 2))
                items.append(plane.rectangle(mat, a, b, float(rng.uniform(-30, 30))))
            elif kind == 3:
                lo = np.array(c)
                items.append(S.Cube(tuple(lo), tuple(lo + rng.uniform(0.5, 8, 3)), mat)
                             .rotate_y(float(rng.uniform(-90, 90))).translate(tuple(rng.uniform(-20, 20, 3))))
            else:
                group = S.List([S.Sphere(tuple(rng.uniform(-5, 5, 3)), 0.5, mat) for _ in range(int(rng.integers(1, 20)))])
                items.append(S.BvhTree(group).translate(c))
        items.append(S.ConstantMedium(S.Cube((0, 0, 0), (3, 3, 3), mat).rotate_y(10.0), 0.2, (1, 1, 1)))
        info = R.flatten_check(S.Scene(S.List(items)).to_desc())
        assert info["records"] >= len(items)


def test_png_roundtrip_and_decoder_vs_pil(tmp_path, earth_rgba):
    from PIL import Image
    mine = R.png_read_rgba8(os.path.join(ROOT, "assets", "earth.png"))
    assert mine.shape == (600, 1200, 4) and np.array_equal(mine, earth_rgba)
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, (37, 53, 4), dtype=np.uint8)
    path = str(tmp_path / "x.png")
    R.png_write_rgba8(path, img)
    assert np.array_equal(np.asarray(Image.open(path).convert("RGBA")), img)  # PIL reads what we write
    assert np.array_equal(R.png_read_rgba8(path), img)
    # PIL-written files with the other colour types / filters decode identically
    for mode in ("RGB", "L", "LA", "P"):
        p2 = str(tmp_path / f"{mode}.png")
        Image.fromarray(img).convert(mode).save(p2, optimize=True)
        assert np.array_equal(R.png_read_rgba8(p2), np.asarray(Image.open(p2).convert("RGBA"))), mode
    with pytest.raises(abi.RtxError):
        R.png_read_rgba8(str(tmp_path / "missing.png"))
    # a missing earth.png is the cyan texture, not an error (texture.rs:96-99)
    d = R.BuiltinDesc(4, earth_png=str(tmp_path / "missing.png"))
    assert not d.desc.images[0].rgba


def test_shard_spp_partitions_exactly():
    for total in (1, 7, 100, 10000):
        for ws in (1, 2, 3, 4, 8):
            parts = [R.shard_spp(total, r, ws) for r in range(ws)]
            assert parts[0][0] == 0 and sum(c for _, c in parts) == total
            for (b0, c0), (b1, _) in zip(parts, parts[1:]):
                assert b0 + c0 == b1
            assert max(c for _, c in parts) - min(c for _, c in parts) <= 1


def test_tile_order_is_a_bijection(tmp_path):
    """kernels.cuh's tile_of_order (the order in which the sample dispenser walks the 8x4-pixel tiles of a frame: blocks
    of 4 x 32 tiles) and order_of_tile are inverse bijections on ragged and very large tile grids (> 2^24 tiles, where the
    float reciprocal needs its correction step) — checked exhaustively by the host program tools/tile_order_check.cu: the
    functions are __host__ __device__, the same code the kernels run."""
    import shutil
    import subprocess
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    exe = tmp_path / "tile_order_check"
    subprocess.run([nvcc, "-std=c++17", "-o", str(exe), os.path.join(ROOT, "tools", "tile_order_check.cu")], check=True, cwd=os.path.join(ROOT, "tools"))
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    assert "bijection on every grid tried" in out


_GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np
import torch, torch.distributed as dist
import rttnw_b200 as R
from tests import _oracle as O
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
rank, world = dist.get_rank(), dist.get_world_size()
# the N > 1 path of bench.py / the CLI with the CPU oracle standing in for the render kernel: every rank builds the
# same scene from the same seed (rtx_builtin_scene / the oracle's own constructor), renders ITS share of the global
# sample indices (R.shard_spp) of every pixel, and one sum-reduce to rank 0 is the whole exchange
W, H, SPP = 24, 16, 13
osc = O.OracleScene.builtin(7)
assert R.flatten_check(R.BuiltinDesc(7))["prim_ids"] == osc.prim_count  # both ranks see the same scene
begin, count = R.shard_spp(SPP, rank, world)
part, rays = osc.render_sum(W, H, count, seed=5, spp_begin=begin, max_depth=4, threads=2)
acc = torch.from_numpy(np.concatenate([part, np.full((H, W, 1), float(count))], axis=2))
dist.reduce(acc, dst=0, op=dist.ReduceOp.SUM)
if rank == 0:
    whole, _ = osc.render_sum(W, H, SPP, seed=5, max_depth=4, threads=2)
    got = acc.numpy()
    assert (got[..., 3] == SPP).all()
    assert np.allclose(got[..., :3], whole, rtol=1e-12, atol=1e-12), np.abs(got[..., :3] - whole).max()
    assert np.array_equal(osc.tonemap(got[..., :3].copy(), SPP), osc.tonemap(whole, SPP))
    print("OK")
dist.destroy_process_group()
"""


def test_spp_sharding_reduce_world_size_2_gloo(tmp_path):
    """Two ranks over gloo: the sharded render (shard_spp over global sample indices + one sum-reduce) equals the
    single-rank render of the same frame, pixel for pixel."""
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / "w.py"
    script.write_text(_GLOO_WORKER.format(root=ROOT, port=port))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
             for r in range(2)]
    outs = [p.communicate(timeout=300) for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert b"OK" in outs[0][0]


def test_ncu_counters_feed_the_bench_line(tmp_path):
    """bench.py turns per-sample ncu counters (tools/r2_counters.py) into live roofline fractions, and refuses
    counters that were captured on other kernel sources."""
    import json
    import bench
    doc = {"kernels_sha": bench.kernels_sha(), "source": "test", "kernels": {
        "wf_trace_kernel": {"warp_instructions_per_sample": 820.0, "lanes_per_warp_instruction": 7.9, "dram_bytes_per_sample": 300.0,
                            "dram_bytes_per_launch": 1.9e7, "l2_bytes_per_sample": 2000.0, "instructions_per_active_sm_cycle": 2.3},
        "wf_shade2_kernel": {"warp_instructions_per_sample": 480.0, "lanes_per_warp_instruction": 13.7, "dram_bytes_per_sample": 500.0,
                             "dram_bytes_per_launch": 3e7, "l2_bytes_per_sample": 3000.0, "instructions_per_active_sm_cycle": 1.6}}}
    r = bench.issue_roof(doc, 600e6, {"sm_mhz": 1965.0}, 148)
    assert abs(r["peak"] - 4 * 148 * 1.965) < 1e-6 and abs(r["achieved"] - 1300 * 0.6) < 1e-6 and 0.5 < r["frac"] < 0.8
    assert abs(r["kernels"]["wf_trace_kernel"]["warp_execution_efficiency"] - 7.9 / 32) < 1e-9
    committed, why = bench.load_counters(9)
    if committed is None:
        assert "no counters" in why or "re-run" in why
    else:
        assert committed["kernels_sha"] == bench.kernels_sha()
        assert any(k.startswith("wf_trace") for k in committed["kernels"]) and any(k.startswith("wf_shade") for k in committed["kernels"])


def test_bench_arms_print_the_same_config():
    """The driver compares the two arms' `config` dicts: they must be equal for the same arguments."""
    import bench
    args = bench.parse.__wrapped__() if hasattr(bench.parse, "__wrapped__") else None
    import argparse
    ns = argparse.Namespace(scene=9, spp=128, width=0, height=0)
    d, w, h = bench.workload(ns)
    assert bench.config(ns, d, w, h) == bench.config(ns, d, w, h)
    assert set(bench.config(ns, d, w, h)) == {"workload", "scene", "width", "height", "spp_per_gpu_per_step", "max_depth", "sharding", "l2"}
    for number in range(1, 10):
        assert bench.scene_defaults(number) == R.scene_defaults(number)  # bench.py's copy of the scene table


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: float32 copies of the arrays, whole while they fit the size limit; past it, one seeded
    sample of pixels, the same on every run and in every array, with its indices."""
    import bench
    rng = np.random.default_rng(3)
    accum = rng.random((50, 40, 4), dtype=np.float32)
    frame = rng.integers(0, 256, (50, 40, 4), dtype=np.uint8)
    bench.dump_outputs(str(tmp_path / "whole"), {"accum": accum, "frame": frame})
    assert sorted(os.listdir(tmp_path / "whole")) == ["accum.npy", "frame.npy"]
    assert np.array_equal(np.load(tmp_path / "whole" / "accum.npy"), accum)
    got = np.load(tmp_path / "whole" / "frame.npy")
    assert got.dtype == np.float32 and np.array_equal(got, frame)
    h, w = 2000, 1500  # 2 x 48 MB as float32: over the limit
    accum = rng.random((h, w, 4), dtype=np.float32)
    frame = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"accum": accum, "frame": frame})
        assert sum(os.path.getsize(tmp_path / run / f) for f in os.listdir(tmp_path / run)) <= bench.DUMP_LIMIT
    idx = np.load(tmp_path / "a" / "pixel_index.npy")
    assert np.array_equal(idx, np.load(tmp_path / "b" / "pixel_index.npy"))
    idx = idx.astype(np.int64)
    assert idx.shape[0] > 0.9 * bench.DUMP_LIMIT / (2 * 16 + 8) and (np.diff(idx) > 0).all() and idx[-1] < h * w
    assert np.array_equal(np.load(tmp_path / "a" / "accum.npy"), accum.reshape(-1, 4)[idx])
    assert np.array_equal(np.load(tmp_path / "a" / "frame.npy"), frame.reshape(-1, 4)[idx])


# ---------------------------------------------------------------------------
# struct layouts: C header (gcc offsetof) == ctypes (abi.py) == Rust #[repr(C)] (ffi.rs), field by field
# ---------------------------------------------------------------------------
_STRUCTS = {"rtx_node": abi.Node, "rtx_material": abi.Material, "rtx_texture": abi.Texture, "rtx_perlin": abi.Perlin,
            "rtx_image": abi.Image, "rtx_camera": abi.Camera, "rtx_scene_desc": abi.SceneDesc, "rtx_ray": abi.Ray,
            "rtx_hit": abi.Hit, "rtx_render_params": abi.RenderParams, "rtx_trace_stats": abi.TraceStats,
            "rtx_scene_defaults": abi.SceneDefaults}


def _rust_layout(src, name):
    """(size, {field: offset}) of a #[repr(C)] struct of ffi.rs under the C layout rules."""
    body = re.search(r"pub struct %s \{(.*?)\n\}" % name, src, re.S).group(1)

    def size_align(t):
        t = t.strip()
        m = re.fullmatch(r"\[(.+); (\d+)\]", t)
        if m:
            s, a = size_align(m.group(1))
            return s * int(m.group(2)), a
        if t.startswith("*const") or t.startswith("*mut"):
            return 8, 8
        if t.startswith("rtx_"):  # a nested struct (all of ours hold an 8-byte member)
            return _rust_layout(src, t)[0], 8
        return {"i32": (4, 4), "u32": (4, 4), "f32": (4, 4), "f64": (8, 8), "u64": (8, 8), "i64": (8, 8), "u8": (1, 1), "usize": (8, 8)}[t]
    off, align, fields = 0, 1, {}
    for fname, ftype in re.findall(r"pub (\w+): ([^,\n]+),", body):
        s, a = size_align(ftype)
        off = (off + a - 1) // a * a
        fields[fname] = off
        off += s
        align = max(align, a)
    return (off + align - 1) // align * align, fields


def test_struct_layouts_header_ctypes_and_rust_agree(tmp_path):
    ffi = open(os.path.join(ROOT, "rust", "rttnw-b200-sys", "src", "ffi.rs")).read()
    # the header's own layout, from the C compiler
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "rttnw_b200.h"', 'int main(void) {']
    for cname, ct in _STRUCTS.items():
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in ct._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    c_layout = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, ct in _STRUCTS.items():
        rsize, rfields = _rust_layout(ffi, cname)
        assert int(c_layout[cname]) == C.sizeof(ct) == rsize, (cname, c_layout[cname], C.sizeof(ct), rsize)
        assert [f for f, _ in ct._fields_] == list(rfields), cname  # same fields in the same order
        for fname, _ in ct._fields_:
            assert int(c_layout[f"{cname}.{fname}"]) == getattr(ct, fname).offset == rfields[fname], (cname, fname)


def test_rust_crate_describes_every_trait_object_of_the_reference():
    """The host crate cannot be compiled here (no Rust toolchain): keep its surface in step with the reference's
    re-exports (src/math/mod.rs:10-19) name by name — every Hittable / Material / Texture has a `describe`."""
    math = open(os.path.join(ROOT, "rust", "rttnw-b200-sys", "src", "math.rs")).read()
    hittables = ["Sphere", "MovingSphere", "List", "BvhTree", "Rectangle<M, P>", "Cube", "Translate", "YRotate", "ConstantMedium"]
    materials = ["Lambertian<T>", "Metal", "Dielectric", "DiffuseLight", "Isotropic"]
    textures = ["Vec3f<Color>", "CheckerTexture", "NoiseTexture", "ImageTexture"]
    for trait, names in (("Hittable", hittables), ("Material", materials), ("Texture", textures)):
        for n in names:
            m = re.search(r"impl(<[^>]*>)? %s for %s \{\s*fn describe" % (trait, re.escape(n)), math)
            assert m, f"math.rs: no `impl {trait} for {n}` with describe"
    for name in ("XY", "XZ", "YZ", "Xy", "Xz", "Yz", "Plane", "Perlin", "CameraDescriptor", "Color", "Position", "Coordinate"):
        assert re.search(r"\b%s\b" % name, math), name
    scenes = open(os.path.join(ROOT, "rust", "rttnw-b200-sys", "src", "scenes.rs")).read()
    assert 'include!(concat!(env!("RTTNW_REFERENCE_SRC"), "/scenes.rs"))' in scenes  # the reference's file, not a copy
    render = open(os.path.join(ROOT, "rust", "rttnw-b200-sys", "src", "render.rs")).read()
    assert "pub fn render(mut width: u32, mut aspect_ratio: f64, mut samples: usize, scene: usize) -> Option<()>" in render
    for n in range(1, 10):
        assert f'"{R.scene_defaults(n)["name"]}"' in render
