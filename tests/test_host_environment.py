"""Environment maps without a GPU: the PFM and Radiance .hdr readers, the ABI surface of rtx_scene_set_environment, and
the oracle's restatement of the lookup (tests/oracle_environment.cpp), whose orientation is pinned here."""
import ctypes as C
import math
import os
import re
import subprocess

import numpy as np
import pytest

import rttnw_b200 as R
from rttnw_b200 import abi
from tests.test_host_cpu import _rust_layout

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTX_ERR_INVALID, RTX_ERR_CUDA, RTX_ERR_IO, RTX_ERR_UNSUPPORTED = -1, -2, -3, -5


# ---------------------------------------------------------------------------
# encoders (the test's own, in numpy)
# ---------------------------------------------------------------------------
def pfm_bytes(img, little=True):
    """PF / Pf, rows bottom-up, scale -1 (little-endian) or +1 (big-endian)."""
    img = np.asarray(img, dtype=np.float32)
    h, w = img.shape[:2]
    head = f"{'PF' if img.ndim == 3 else 'Pf'}\n{w} {h}\n{-1.0 if little else 1.0}\n".encode()
    return head + np.ascontiguousarray(img[::-1]).astype("<f4" if little else ">f4").tobytes()


def rgbe(rgb):
    """(H, W, 4) uint8 RGBE of float texels, and the floats they decode to: m * 2^(e - 136)."""
    rgb = np.asarray(rgb, dtype=np.float64)
    mx = rgb.max(axis=-1)
    out = np.zeros(rgb.shape[:2] + (4,), dtype=np.uint8)
    nz = mx > 1e-32
    m, e = np.frexp(mx[nz])  # mx = m 2^e, m in [0.5, 1)
    out[nz, :3] = np.floor(rgb[nz] * (256.0 / mx[nz])[:, None] * m[:, None]).clip(0, 255).astype(np.uint8)
    out[nz, 3] = (e + 128).astype(np.uint8)
    dec = np.where(out[..., 3:] == 0, 0.0, out[..., :3] * np.exp2(out[..., 3:].astype(np.float64) - 136.0))
    return out, dec.astype(np.float32)


def rle_channel(v):
    """New-style run-length encoding of one component of a scanline: runs of >= 3 equal bytes, else literals."""
    out, i, n = bytearray(), 0, len(v)
    while i < n:
        j = i
        while j < n and j - i < 127 and v[j] == v[i]:
            j += 1
        if j - i >= 3:
            out += bytes([128 + j - i, v[i]])
            i = j
            continue
        k = i
        while k < n and k - i < 128 and not (k + 2 < n and v[k] == v[k + 1] == v[k + 2]):
            k += 1
        out += bytes([k - i]) + bytes(v[i:k])
        i = k
    return bytes(out)


def hdr_bytes(px, rle, resolution=None, fmt="32-bit_rle_rgbe"):
    h, w = px.shape[:2]
    head = f"#?RADIANCE\n# written by a test\nFORMAT={fmt}\n\n{resolution or f'-Y {h} +X {w}'}\n".encode()
    body = bytearray()
    for y in range(h):
        if rle:
            body += bytes([2, 2, w >> 8, w & 255])
            for c in range(4):
                body += rle_channel(px[y, :, c].tolist())
        else:
            body += px[y].tobytes()
    return head + bytes(body)


def smooth_map(h, w, seed):
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w]
    base = 0.5 + 0.4 * np.sin(x[..., None] * 2 * np.pi / w + rng.random(3) * 6) * np.cos(y[..., None] * np.pi / h)
    base[h // 3, w // 4:w // 2] = 0.0  # runs of zeros and of equal texels exercise both RLE forms
    base[1, :] = 3.0
    return base.astype(np.float32)


def read_status(fn, path):
    lib = abi.load()
    w, h, c, buf = C.c_int32(), C.c_int32(), C.c_int32(), C.POINTER(C.c_float)()
    if fn == "pfm":
        rc = lib.rtx_pfm_read(str(path).encode(), C.byref(w), C.byref(h), C.byref(c), C.byref(buf))
    else:
        rc = lib.rtx_hdr_read(str(path).encode(), C.byref(w), C.byref(h), C.byref(buf))
    if rc == 0:
        lib.rtx_buffer_free(buf)
    return rc


# ---------------------------------------------------------------------------
# PFM
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(1, 1, 3), (5, 7, 3), (33, 64, 3), (4, 9)])
def test_pfm_round_trip_through_the_writer(tmp_path, shape):
    img = np.random.default_rng(3).standard_normal(shape).astype(np.float32) * 100
    img.flat[0] = np.float32(np.inf)  # the reader returns bits, it does not judge them
    R.pfm_write(str(tmp_path / "a.pfm"), img)
    back = R.pfm_read(str(tmp_path / "a.pfm"))
    assert back.shape == img.shape and back.dtype == np.float32 and back.tobytes() == img.tobytes()


@pytest.mark.parametrize("little", [True, False])
def test_pfm_both_byte_orders(tmp_path, little):
    img = smooth_map(6, 10, 1)
    (tmp_path / "a.pfm").write_bytes(pfm_bytes(img, little))
    assert R.pfm_read(str(tmp_path / "a.pfm")).tobytes() == img.tobytes()
    grey = img[..., 1]
    (tmp_path / "g.pfm").write_bytes(pfm_bytes(grey, little))
    assert R.pfm_read(str(tmp_path / "g.pfm")).tobytes() == grey.tobytes()
    assert np.array_equal(R.env_read(str(tmp_path / "g.pfm")), np.repeat(grey[..., None], 3, axis=2))


# ---------------------------------------------------------------------------
# Radiance .hdr
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("rle, w", [(False, 5), (False, 8), (False, 300), (True, 8), (True, 300)])  # (RLE needs w >= 8)
def test_hdr_flat_and_rle_read_back_exactly(tmp_path, rle, w):
    px, want = rgbe(smooth_map(7, w, w) * np.array([1.0, 20.0, 1e-3], dtype=np.float32))
    (tmp_path / "a.hdr").write_bytes(hdr_bytes(px, rle))
    got = R.hdr_read(str(tmp_path / "a.hdr"))
    assert got.shape == (7, w, 3) and got.tobytes() == want.tobytes()
    assert np.array_equal(R.env_read(str(tmp_path / "a.hdr")), want)


def test_hdr_other_orientations_are_unsupported(tmp_path):
    px, _ = rgbe(smooth_map(4, 8, 2))
    for res in ("+Y 4 +X 8", "-Y 4 -X 8", "+X 8 -Y 4", "-X 8 +Y 4"):
        (tmp_path / "a.hdr").write_bytes(hdr_bytes(px, False, res))
        assert read_status("hdr", tmp_path / "a.hdr") == RTX_ERR_UNSUPPORTED, res
    (tmp_path / "b.hdr").write_bytes(hdr_bytes(px, False, fmt="32-bit_rle_xyze"))
    assert read_status("hdr", tmp_path / "b.hdr") == RTX_ERR_UNSUPPORTED


def test_truncated_and_malformed_files_give_an_error(tmp_path):
    """Every prefix of a valid file, and a set of broken headers and runs, is refused with RTX_ERR_INVALID: never a
    crash or an over-read (the library reads the file into a buffer of its exact size)."""
    img = smooth_map(5, 12, 4)
    px, _ = rgbe(img)
    files = {"pfm": pfm_bytes(img), "hdr": hdr_bytes(px, True), "hdr_flat": hdr_bytes(px, False)}
    for kind, data in files.items():
        fn = "pfm" if kind == "pfm" else "hdr"
        for n in range(len(data)):
            (tmp_path / "t").write_bytes(data[:n])
            assert read_status(fn, tmp_path / "t") == RTX_ERR_INVALID, (kind, n)
        (tmp_path / "t").write_bytes(data)
        assert read_status(fn, tmp_path / "t") == 0
    bad_pfm = [b"PX\n2 2\n-1\n" + bytes(48), b"PF\n0 2\n-1\n", b"PF\n2 -2\n-1\n" + bytes(48), b"PF\n2 2\n0\n" + bytes(48),
               b"PF\n2 2\nnan\n" + bytes(48), b"PF\n99999999 99999999\n-1\n" + bytes(64), b"PF\n2 2\n-1" + bytes(48)[:0]]
    for data in bad_pfm:
        (tmp_path / "b").write_bytes(data)
        assert read_status("pfm", tmp_path / "b") == RTX_ERR_INVALID, data[:24]
    head = b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n-Y 1 +X 8\n"
    bad_hdr = [b"P6\n", b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n", b"#?RADIANCE\n\n-Y x +X 8\n" + bytes(32),
               b"#?RADIANCE\n\n-Y 1 +X 8 extra\n" + bytes(32), b"#?RADIANCE\n\n-Y 0 +X 8\n",
               head + bytes([2, 2, 0, 8]) + bytes([0]),                      # a literal run of length 0
               head + bytes([2, 2, 0, 8]) + bytes([9]) + bytes(9),           # a literal run past the scanline
               head + bytes([2, 2, 0, 8]) + bytes([128 + 9, 1]),             # a repeat run past the scanline
               head + bytes([2, 2, 0, 8]) + bytes([128 + 8])]                 # a repeat run without its byte
    for data in bad_hdr:
        (tmp_path / "b").write_bytes(data)
        assert read_status("hdr", tmp_path / "b") == RTX_ERR_INVALID, data
    assert read_status("pfm", tmp_path / "missing.pfm") == RTX_ERR_IO
    assert read_status("hdr", tmp_path / "missing.hdr") == RTX_ERR_IO
    (tmp_path / "x.png").write_bytes(b"\x89PNG....")
    with pytest.raises(ValueError):
        R.env_read(str(tmp_path / "x.png"))


# ---------------------------------------------------------------------------
# the ABI surface
# ---------------------------------------------------------------------------
def test_environment_struct_layout_header_ctypes_and_rust_agree(tmp_path):
    ffi = open(os.path.join(ROOT, "rust", "rttnw-b200-sys", "src", "ffi.rs")).read()
    fields = [f for f, _ in abi.Environment._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "rttnw_b200.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(rtx_environment));']
    lines += [f'  printf("{f} %zu\\n", offsetof(rtx_environment, {f}));' for f in fields] + ['  return 0;', '}']
    (tmp_path / "l.c").write_text("\n".join(lines))
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(tmp_path / "l.c"), "-o", str(tmp_path / "l")], check=True)
    c = dict(l.split() for l in subprocess.run([str(tmp_path / "l")], check=True, capture_output=True, text=True).stdout.splitlines())
    rsize, rfields = _rust_layout(ffi, "rtx_environment")
    assert int(c["size"]) == C.sizeof(abi.Environment) == rsize == 48
    assert list(rfields) == fields
    for f in fields:
        assert int(c[f]) == getattr(abi.Environment, f).offset == rfields[f], f


def test_new_symbols_are_in_the_library_and_the_rust_bindings():
    lib = abi.load()
    ffi = open(os.path.join(ROOT, "rust", "rttnw-b200-sys", "src", "ffi.rs")).read()
    lib_rs = open(os.path.join(ROOT, "rust", "rttnw-b200-sys", "src", "lib.rs")).read()
    for name in ("rtx_scene_set_environment", "rtx_pfm_read", "rtx_hdr_read"):
        assert hasattr(lib, name) and name in abi.SIGNATURES
        assert re.search(r"pub fn %s\(" % name, ffi), name
    assert "pub fn set_environment(" in lib_rs


def test_the_new_calls_fail_loudly_without_a_device():
    """A NULL context or scene is refused before anything else; without a CUDA device no context (so no scene) can
    exist, and creating one fails with RTX_ERR_CUDA like every compute entry point."""
    lib = abi.load()
    rgb = np.ones(3, dtype=np.float32)
    env = abi.Environment(1, 1, rgb.ctypes.data_as(C.POINTER(C.c_float)), 0.0, (C.c_double * 3)(1, 1, 1))
    assert lib.rtx_scene_set_environment(None, None, C.byref(env)) == RTX_ERR_INVALID
    assert lib.rtx_scene_set_environment(None, None, None) == RTX_ERR_INVALID
    n = C.c_int(0)
    if lib.rtx_device_count(C.byref(n)) != 0 or n.value == 0:
        h = C.c_void_p()
        assert lib.rtx_ctx_create(0, None, C.byref(h)) == RTX_ERR_CUDA
        assert b"" != lib.rtx_last_error()


# ---------------------------------------------------------------------------
# the oracle's lookup: the convention of the header, pinned on known directions
# ---------------------------------------------------------------------------
def oracle_env_lib(tmp_path_factory):
    mk = open(os.path.join(ROOT, "oracle", "Makefile")).read()
    flags = re.search(r"^CXXFLAGS \?= (.*)$", mk, re.M).group(1).split()
    out = tmp_path_factory.mktemp("oracle_environment") / "liboracle_environment.so"
    subprocess.run([os.environ.get("CXX", "g++"), *flags, "-shared", "-o", str(out),
                    os.path.join(ROOT, "tests", "oracle_environment.cpp"), "-lpthread"], check=True, capture_output=True)
    lib = C.CDLL(str(out))
    sig = {"orc_scene_builtin": (C.c_void_p, [C.c_int, C.c_uint64, C.c_void_p, C.c_int, C.c_int]),
           "orc_scene_from_desc": (C.c_void_p, [C.POINTER(abi.SceneDesc), C.c_uint64]),
           "orc_scene_free": (None, [C.c_void_p]),
           "orc_scene_set_environment": (None, [C.c_void_p, C.POINTER(abi.Environment)]),
           "orc_environment_value": (None, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
           "orc_render_env": (C.c_uint64, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_void_p,
                                           C.c_int]),
           "orc_first_vertex_env": (None, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_int])}
    for name, (res, args) in sig.items():
        getattr(lib, name).restype, getattr(lib, name).argtypes = res, args
    return lib


@pytest.fixture(scope="module")
def env_lib(tmp_path_factory):
    return oracle_env_lib(tmp_path_factory)


def sector_map(w=64, h=32):
    """Columns in four sectors centred on u = 0, 0.25, 0.5, 0.75 and rows in three bands (top quarter, middle, bottom
    quarter): a colour per (band, sector) in the middle band, one colour per polar band."""
    u = (np.arange(w) + 0.5) / w
    sector = np.floor(4 * u + 0.5).astype(int) % 4
    v = (np.arange(h) + 0.5) / h
    band = np.where(v < 0.25, 0, np.where(v > 0.75, 2, 1))
    colours = {(1, s): np.array([0.1 + 0.2 * s, 0.9 - 0.2 * s, 0.5], dtype=np.float32) for s in range(4)}
    img = np.zeros((h, w, 3), dtype=np.float32)
    for j in range(h):
        for i in range(w):
            img[j, i] = colours[(1, sector[i])] if band[j] == 1 else ([2.0, 2.0, 2.0] if band[j] == 0 else [0.0, 0.0, 0.25])
    return img, colours


# direction -> (band, sector) at rotation 0 and at rotation 90 (the centre column, u = 0.5, seen along -z and -x)
AXES = {(0, 0, -1): ((1, 2), (1, 3)), (1, 0, 0): ((1, 3), (1, 0)), (0, 0, 1): ((1, 0), (1, 1)), (-1, 0, 0): ((1, 1), (1, 2)),
        (0, 1, 0): ((0, None), (0, None)), (0, -1, 0): ((2, None), (2, None))}


def expected_colour(img, colours, key):
    band, sector = key
    return colours[(1, sector)] if band == 1 else (img[0, 0] if band == 0 else img[-1, 0])


def set_oracle_env(lib, h, img, rotation=0.0, scale=(1.0, 1.0, 1.0)):
    img = np.ascontiguousarray(img, dtype=np.float32)
    env = abi.Environment(img.shape[1], img.shape[0], img.ctypes.data_as(C.POINTER(C.c_float)), rotation,
                          (C.c_double * 3)(*scale))
    lib.orc_scene_set_environment(h, C.byref(env))


def test_oracle_lookup_orientation(env_lib):
    """Along the axes the sector map gives back the sector the header's convention names, not mirrored, at rotation
    0 and 90; a 1x1 map gives its value for any direction; scale multiplies; removing the map gives the background."""
    desc = R.BuiltinDesc(2)
    h = env_lib.orc_scene_from_desc(C.byref(desc.desc), 7)
    img, colours = sector_map()
    for k, rot in enumerate((0.0, 90.0)):
        set_oracle_env(env_lib, h, img, rot)
        dirs = np.array([d for d in AXES], dtype=np.float64) * 3.0  # not normalised
        out = np.zeros_like(dirs)
        env_lib.orc_environment_value(h, len(dirs), dirs.ctypes.data, out.ctypes.data)
        for d, got in zip(AXES, out):
            assert np.allclose(got, expected_colour(img, colours, AXES[d][k]), rtol=0, atol=1e-12), (rot, d, got)
    one = np.array([[[0.3, 1.7, 42.0]]], dtype=np.float32)
    set_oracle_env(env_lib, h, one, 123.0, (2.0, 0.5, 1.0))
    dirs = np.random.default_rng(5).standard_normal((1000, 3))
    out = np.zeros_like(dirs)
    env_lib.orc_environment_value(h, len(dirs), dirs.ctypes.data, out.ctypes.data)
    assert np.array_equal(out, np.broadcast_to(one[0, 0].astype(np.float64) * [2.0, 0.5, 1.0], out.shape))
    env_lib.orc_scene_set_environment(h, None)
    env_lib.orc_environment_value(h, 1, dirs.ctypes.data, out.ctypes.data)
    assert np.array_equal(out[0], list(desc.desc.background))
    env_lib.orc_scene_free(h)


def test_oracle_lookup_blends_bilinearly(env_lib):
    """u and v of a direction, then the texel coordinates: a direction at a texel centre gives that texel, and halfway
    between two centres of one row their mean; columns wrap across the seam."""
    desc = R.BuiltinDesc(2)
    h = env_lib.orc_scene_from_desc(C.byref(desc.desc), 7)
    w_, h_ = 16, 8
    img = np.random.default_rng(9).random((h_, w_, 3)).astype(np.float32)
    set_oracle_env(env_lib, h, img)

    def direction(u, v):  # the inverse of the header's mapping at rotation 0
        phi, theta = (u - 0.5) * 2 * math.pi, v * math.pi
        return [math.sin(theta) * math.sin(phi), math.cos(theta), -math.sin(theta) * math.cos(phi)]

    cases = [((i + 0.5) / w_, (j + 0.5) / h_, img[j, i]) for i, j in ((3, 2), (0, 5), (15, 4))]
    cases.append(((4.0 + 0.5 + 0.5) / w_, 3.5 / h_, (img[3, 4].astype(np.float64) + img[3, 5]) / 2))
    cases.append((0.0 + 1e-9, 2.5 / h_, (img[2, 0].astype(np.float64) + img[2, 15]) / 2))  # the seam
    dirs = np.array([direction(u, v) for u, v, _ in cases])
    out = np.zeros_like(dirs)
    env_lib.orc_environment_value(h, len(dirs), dirs.ctypes.data, out.ctypes.data)
    for (u, v, want), got in zip(cases, out):
        assert np.allclose(got, want, rtol=0, atol=1e-6), (u, v, got, want)
    env_lib.orc_scene_free(h)
