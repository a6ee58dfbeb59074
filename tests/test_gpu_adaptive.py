"""Adaptive sampling (rtx_render_adaptive, rtx_adaptive_error), checked path by path.

Every random draw is Philox keyed by (pixel, global sample index, bounce), so an adaptive frame, in which each 8x4 tile
of pixels ends with the samples [spp_begin, spp_begin + n) of the uniform render, can be compared pixel by pixel with
the single-path radiances of test_gpu_render_paths.gpu_paths: accum.rgb must be the sum of the pixel's first n paths
and aux.rgb the sum of those with an odd index, within the fp32 summation-order bound n * 2^-24 * sum |x| (the paths are
fp32 values; the accumulators add them with atomics in no fixed order). The stopping rule is recomputed from the outside
with rtx_adaptive_error on uniform prefix sums of the same paths; a tile whose error lies within 1e-4 relative of the
threshold may fall either way (the render's own sums differ from the prefix sums in the last bits).
"""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import rttnw_b200 as R
from rttnw_b200 import abi
from tests import _oracle as O
from tests._record import record

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, H = 96, 72
MIN, STEP, MAX = 8, 8, 64
U = 2.0 ** -24
NEAR = 1e-4  # relative distance to the threshold inside which a tile may fall either way


@pytest.fixture(scope="module")
def ctx():
    c = R.Context(0)
    yield c
    c.close()


# ---------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------
def adaptive(gsc, thr, mn, st, mx, seed, depth=50, begin=0, w=W, h=H):
    acc, aux = gsc.new_accum(w, h), gsc.new_accum(w, h)
    stats = gsc.render_adaptive(acc, aux, thr, mn, st, mx, seed=seed, max_depth=depth, spp_begin=begin)
    return acc.cpu().numpy().astype(np.float64), aux.cpu().numpy().astype(np.float64), stats


def prefix_sums(paths, begin=0):
    """(S+1, H, W, 3) sums of the first n paths and of the odd-indexed ones among them (global index begin + k)."""
    odd = ((begin + np.arange(paths.shape[0])) % 2 == 1)[:, None, None, None]
    z = np.zeros((1,) + paths.shape[1:])
    return np.concatenate([z, np.cumsum(paths, axis=0)]), np.concatenate([z, np.cumsum(paths * odd, axis=0)])


def tile_errors(gsc, paths, ns, begin=0):
    """n -> (tiles_y, tiles_x) error of the uniform prefix of n samples, from rtx_adaptive_error."""
    torch = gsc.ctx.torch
    full, odd = prefix_sums(paths, begin)
    h, w = paths.shape[1:3]
    out = {}
    for n in ns:
        a = np.concatenate([full[n], np.full((h, w, 1), n)], axis=-1).astype(np.float32)
        b = np.concatenate([odd[n], np.full((h, w, 1), n // 2)], axis=-1).astype(np.float32)
        da, db = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
        out[n] = gsc.adaptive_error(da, db).cpu().numpy().astype(np.float64)
    return out


def simulate(err, thr, mn, st, mx):
    """The stopping rule on precomputed errors: n per tile."""
    n = np.full(err[mn].shape, mn)
    active = np.ones(err[mn].shape, dtype=bool)
    cur = mn
    while cur < mx:
        active &= ~(err[cur] < thr)
        if not active.any():
            break
        cur = min(cur + st, mx)
        n[active] = cur
    return n


def mix(n, mn, mx):
    return float((n == mn).mean()), float(((n > mn) & (n < mx)).mean()), float((n == mx).mean())


def pick_threshold(err, mn, st, mx):
    """From the 8-spp error map's quantiles, the threshold whose simulated tile counts are most evenly mixed."""
    best = None
    for q in np.linspace(0.05, 0.9, 35):
        thr = float(np.quantile(err[mn], q))
        score = min(mix(simulate(err, thr, mn, st, mx), mn, mx))
        if best is None or score > best[0]:
            best = (score, thr)
    return best[1]


def tile_n(acc):
    """n per tile (top-left pixel), after checking that every pixel of a tile has it."""
    h, w = acc.shape[:2]
    n = acc[..., 3]
    ty, tx = np.arange(h) // 4, np.arange(w) // 8
    per_tile = n[::4, ::8]
    assert (n == per_tile[ty][:, tx]).all(), "pixels of one tile differ in their sample count"
    return per_tile.astype(np.int64)


def check_prefix(acc, aux, paths, begin=0):
    """accum / aux against the sums of each pixel's own prefix of single paths, within the summation bound."""
    n = acc[..., 3].astype(np.int64)
    assert (aux[..., 3] == n // 2).all()
    full, odd = prefix_sums(paths, begin)
    iy, ix = np.indices(n.shape)
    want, want_odd = full[n, iy, ix], odd[n, iy, ix]
    bound = n[..., None] * U * want  # paths are >= 0: sum |x| is the sum
    bound_odd = (n // 2)[..., None] * U * want_odd
    assert (np.abs(acc[..., :3] - want) <= bound).all(), np.abs(acc[..., :3] - want).max()
    assert (np.abs(aux[..., :3] - want_odd) <= bound_odd).all(), np.abs(aux[..., :3] - want_odd).max()


def check_stopping(n, err, thr, mn, st, mx):
    """Every tile's n follows from the errors of the uniform prefixes. Returns how many decisions were exempt."""
    near = 0

    def below(e):
        nonlocal near
        if abs(e - thr) <= NEAR * thr:
            near += 1
            return None  # either way
        return e < thr

    for (y, x), k in np.ndenumerate(n):
        if k < mx:  # stopped below the threshold at k
            assert below(err[k][y, x]) in (True, None), ((y, x), k, err[k][y, x], thr)
        if k > mn:  # and kept going at the round before
            prev = max(mn, k - st) if k < mx else mn + (mx - mn - 1) // st * st
            assert below(err[prev][y, x]) in (False, None), ((y, x), k, prev, err[prev][y, x], thr)
    return near


def check_stats(stats, acc, mn, st, mx):
    n = tile_n(acc)
    assert stats["path_samples"] == int(acc[..., 3].sum())
    assert stats["tiles"] == n.size
    assert stats["tiles_at_max"] == int((n == mx).sum())
    assert stats["tiles_converged"] == int((n < mx).sum())
    top = int(n.max())
    assert stats["rounds"] == 1 + math.ceil((top - mn) / st)


_CASES = {}


def prefix_case(ctx, number):
    """Scene `number` at min 8 / step 8 / max 64: the single paths, the prefix errors, the threshold and the frame."""
    if number not in _CASES:
        from tests.test_gpu_render_paths import gpu_paths
        gsc = R.DeviceScene(ctx, R.BuiltinDesc(number))
        seed = 40 + number
        paths = gpu_paths(gsc, W, H, MAX, seed, 50)
        err = tile_errors(gsc, paths, range(MIN, MAX + 1, STEP))
        thr = pick_threshold(err, MIN, STEP, MAX)
        acc, aux, stats = adaptive(gsc, thr, MIN, STEP, MAX, seed)
        _CASES[number] = dict(gsc=gsc, seed=seed, paths=paths, err=err, thr=thr, acc=acc, aux=aux, stats=stats)
    return _CASES[number]


# ---------------------------------------------------------------------------
# 1, 4, 8: prefix property, stopping rule and stats on scenes 3, 7 and 9
# ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("number", [3, 7, 9])
def test_every_pixel_holds_a_prefix_of_the_uniform_render(ctx, number):
    c = prefix_case(ctx, number)
    n = tile_n(c["acc"])
    shares = mix(n, MIN, MAX)
    record("adaptive", f"prefix_scene_{number}", {"threshold": c["thr"], "share_at_min": shares[0], "share_between": shares[1],
                                                  "share_at_max": shares[2], "stats": c["stats"]})
    assert min(shares) >= 0.10, shares
    assert set(np.unique(n)) <= set(range(MIN, MAX + 1, STEP))
    check_prefix(c["acc"], c["aux"], c["paths"])


@pytest.mark.gpu
@pytest.mark.parametrize("number", [3, 7, 9])
def test_stopping_rule_recomputed_from_uniform_prefixes(ctx, number):
    c = prefix_case(ctx, number)
    n = tile_n(c["acc"])
    near = check_stopping(n, c["err"], c["thr"], MIN, STEP, MAX)
    record("adaptive", f"stopping_scene_{number}", {"tiles": int(n.size), "decisions_within_1e-4_of_threshold": near})
    assert near <= 0.05 * n.size, near


@pytest.mark.gpu
@pytest.mark.parametrize("number", [3, 7, 9])
def test_stats_match_the_buffers(ctx, number):
    c = prefix_case(ctx, number)
    check_stats(c["stats"], c["acc"], MIN, STEP, MAX)


# ---------------------------------------------------------------------------
# 2: oracle, per pixel over its own prefix
# ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("number,depth", [(7, 2), (9, 50)])
def test_adaptive_sums_match_the_oracle(ctx, number, depth, earth_rgba):
    from tests.test_gpu_render_paths import MIN_AGREE, Z_MAX, compare_paths, gpu_paths, scene_tolerance
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(number))
    osc = O.OracleScene.builtin(number, earth=earth_rgba)
    seed = 60 + number
    err = tile_errors(gsc, gpu_paths(gsc, W, H, MAX, seed, depth), range(MIN, MAX + 1, STEP))
    thr = pick_threshold(err, MIN, STEP, MAX)
    acc, aux, _ = adaptive(gsc, thr, MIN, STEP, MAX, seed, depth=depth)
    n = acc[..., 3].astype(np.int64)
    ref = np.stack([osc.render_sum(W, H, 1, seed=seed, spp_begin=k, max_depth=depth)[0] for k in range(MAX)])
    full, _ = prefix_sums(ref)
    iy, ix = np.indices(n.shape)
    want = full[n, iy, ix]
    rtol, atol = scene_tolerance(number)
    st = compare_paths(acc[..., :3], want, rtol, atol * n[..., None])
    st["atol"] = f"{atol} per sample"
    st["min_share_allowed"] = MIN_AGREE[(number, depth)]
    st["mix"] = mix(tile_n(acc), MIN, MAX)
    record("adaptive", f"oracle_scene_{number}_depth_{depth}", st)
    assert st["agree_share"] >= st["min_share_allowed"], st
    assert max(st["z"]) <= Z_MAX, st


# ---------------------------------------------------------------------------
# 3: the error kernel against a float64 restatement
# ---------------------------------------------------------------------------
def error_reference(acc, aux):
    h, w = acc.shape[:2]
    a, b = acc.astype(np.float64), aux.astype(np.float64)
    ok = (a[..., 3] > 0) & (b[..., 3] > 0)
    with np.errstate(all="ignore"):
        i = a[..., :3] / a[..., 3:4]
        m = b[..., :3] / b[..., 3:4]
        e = np.abs(i - m).sum(axis=-1) / (1e-4 + np.sqrt(i.sum(axis=-1)))
    e = np.where(ok, e, 0.0)
    ty, tx = (h + 3) // 4, (w + 7) // 8
    pad = np.zeros((ty * 4, tx * 8))
    pad[:h, :w] = e
    return pad.reshape(ty, 4, tx, 8).max(axis=(1, 3))


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(1, 1), (7, 3), (33, 17), (96, 72)])
def test_error_kernel_matches_a_float64_restatement(ctx, w, h):
    import torch
    rng = np.random.default_rng(w * 100 + h)
    n = rng.choice([2, 8, 64, 1000], size=(h, w)).astype(np.float32)
    acc = np.concatenate([rng.random((h, w, 3)) * n[..., None], n[..., None]], axis=-1).astype(np.float32)
    aux = np.concatenate([rng.random((h, w, 3)) * (n / 2)[..., None], (n / 2)[..., None]], axis=-1).astype(np.float32)
    if w * h >= 32:
        acc[:4, :8, :3] = 0.0  # a tile of black pixels in both halves: error 0
        aux[:4, :8, :3] = 0.0
        acc[min(5, h - 1), min(9, w - 1), :3] *= 50.0  # one hot pixel sets its tile's error
    da, db = torch.from_numpy(acc).cuda(), torch.from_numpy(aux).cuda()
    d_err = torch.full(((h + 3) // 4, (w + 7) // 8), -1.0, device="cuda")
    abi.check(ctx.lib.rtx_adaptive_error(ctx.h, da.data_ptr(), db.data_ptr(), w, h, d_err.data_ptr()))
    got = d_err.cpu().numpy()
    want = error_reference(acc, aux)
    assert got.shape == want.shape == ((h + 3) // 4, (w + 7) // 8)
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=0)
    if w * h >= 32:
        assert got[0, 0] == 0.0
        y, x = min(5, h - 1) // 4, min(9, w - 1) // 8
        pix = error_reference(acc[y * 4:y * 4 + 4, x * 8:x * 8 + 8], aux[y * 4:y * 4 + 4, x * 8:x * 8 + 8])
        assert got[y, x] == pytest.approx(float(pix.max()), rel=1e-5)


# ---------------------------------------------------------------------------
# 5: edge cases
# ---------------------------------------------------------------------------
@pytest.mark.gpu
def test_threshold_zero_is_the_uniform_render(ctx):
    from tests.test_gpu_render_paths import gpu_paths
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(7))
    paths = gpu_paths(gsc, W, H, 16, 71, 50)
    acc, aux, stats = adaptive(gsc, 0.0, 4, 4, 16, 71)
    assert (acc[..., 3] == 16).all() and stats["tiles_at_max"] == stats["tiles"] and stats["rounds"] == 4
    uni = gsc.new_accum(W, H)
    gsc.render_into(uni, 0, 16, seed=71)
    uni = uni.cpu().numpy().astype(np.float64)
    bound = 2 * 16 * U * paths.sum(axis=0)
    assert (np.abs(acc[..., :3] - uni[..., :3]) <= bound).all()
    check_prefix(acc, aux, paths)


@pytest.mark.gpu
def test_huge_threshold_stops_every_tile_at_min(ctx):
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(9))
    acc, aux, stats = adaptive(gsc, 1e30, 6, 4, 64, 5)
    assert (acc[..., 3] == 6).all() and (aux[..., 3] == 3).all()
    assert stats["rounds"] == 1 and stats["tiles_converged"] == stats["tiles"] and stats["path_samples"] == 6 * W * H


@pytest.mark.gpu
def test_min_equal_to_max(ctx):
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(7))
    acc, _, stats = adaptive(gsc, 1e-3, 8, 2, 8, 5)
    assert (acc[..., 3] == 8).all() and stats["rounds"] == 1 and stats["tiles_at_max"] == stats["tiles"]


@pytest.mark.gpu
def test_shorter_last_round_and_an_offset_begin(ctx):
    """max 14 with step 6 from min 4: rounds of 4, 6 and 4 samples; the samples are the global indices [6, 20)."""
    from tests.test_gpu_render_paths import gpu_paths
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(9))
    paths = gpu_paths(gsc, W, H, 14, 9, 50, begin=6)
    acc, aux, stats = adaptive(gsc, 0.0, 4, 6, 14, 9, begin=6)
    assert (acc[..., 3] == 14).all() and stats["rounds"] == 3
    check_prefix(acc, aux, paths, begin=6)
    check_stats(stats, acc, 4, 6, 14)


@pytest.mark.gpu
def test_depth_zero_moves_only_the_counts(ctx):
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(9))
    acc, aux, stats = adaptive(gsc, 0.01, 4, 4, 16, 3, depth=0, w=33, h=17)
    assert (acc[..., :3] == 0).all() and (aux[..., :3] == 0).all()
    assert (acc[..., 3] == 4).all() and (aux[..., 3] == 2).all()
    assert stats["rounds"] == 1 and stats["tiles"] == 5 * 5 and stats["tiles_converged"] == 25
    assert stats["path_samples"] == 4 * 33 * 17


def _call(ctx, gsc, w=W, h=H, begin=0, mx=16, thr=0.01, mn=4, st=4, aux=True):
    torch = ctx.torch
    acc = torch.zeros((max(h, 1), max(w, 1), 4), dtype=torch.float32, device="cuda")
    ax = torch.zeros_like(acc)
    p = abi.RenderParams(w, h, begin, mx, 50, 0, 1)
    ap = abi.AdaptiveParams(thr, mn, st)
    return ctx.lib.rtx_render_adaptive(ctx.h, gsc.h, C.byref(p), C.byref(ap), acc.data_ptr(),
                                       ax.data_ptr() if aux else None, None)


@pytest.mark.gpu
def test_invalid_arguments_are_refused(ctx):
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(7))
    bad = [dict(mx=15), dict(mx=0), dict(mx=2 ** 24 + 2), dict(mn=3), dict(mn=0), dict(mn=18), dict(st=3), dict(st=0),
           dict(thr=-1e-9), dict(thr=float("nan")), dict(thr=float("inf")), dict(begin=1), dict(aux=False), dict(w=0),
           dict(h=-4)]
    for kw in bad:
        assert _call(ctx, gsc, **kw) == -1, kw
    assert _call(ctx, gsc) == 0
    lib = ctx.lib
    import torch
    a = torch.zeros((4, 8, 4), device="cuda")
    out = torch.zeros((1, 1), device="cuda")
    assert lib.rtx_adaptive_error(ctx.h, a.data_ptr(), None, 8, 4, out.data_ptr()) == -1
    assert lib.rtx_adaptive_error(ctx.h, a.data_ptr(), a.data_ptr(), 0, 4, out.data_ptr()) == -1


@pytest.mark.gpu
@pytest.mark.parametrize("setting", ["RTX_SHADE=1", "RTX_MODE=mega", "RTX_ORDER=1"])
def test_unsupported_driver_forms_are_refused(setting, monkeypatch):
    k, v = setting.split("=")
    monkeypatch.setenv(k, v)
    c = R.Context(0)
    try:
        gsc = R.DeviceScene(c, R.BuiltinDesc(7))
        assert _call(c, gsc) == -5
        gsc.close()
    finally:
        c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("setting", ["RTX_TRACE=2", "RTX_TRACE=3", "RTX_TRACE=4", "RTX_BVH_WIDE=1"])
def test_other_trace_forms_keep_the_prefix_property(setting, ctx, monkeypatch):
    c = prefix_case(ctx, 9)
    k, v = setting.split("=")
    monkeypatch.setenv(k, v)
    c2 = R.Context(0)
    try:
        gsc = R.DeviceScene(c2, R.BuiltinDesc(9))
        acc, aux, stats = adaptive(gsc, c["thr"], MIN, STEP, MAX, c["seed"])
        check_prefix(acc, aux, c["paths"])
        check_stats(stats, acc, MIN, STEP, MAX)
        assert min(mix(tile_n(acc), MIN, MAX)) >= 0.05
        gsc.close()
    finally:
        c2.close()


# ---------------------------------------------------------------------------
# 6, 7: no state leaks into the next plain render; the tonemap divides by each pixel's own count
# ---------------------------------------------------------------------------
@pytest.mark.gpu
def test_plain_render_after_adaptive_is_unchanged():
    def plain(c):
        gsc = R.DeviceScene(c, R.BuiltinDesc(9))
        acc = gsc.new_accum(W, H)
        gsc.render_into(acc, 0, 1, seed=13)
        c.sync()
        out = acc.cpu().numpy().tobytes()
        gsc.close()
        return out
    c1 = R.Context(0)
    try:
        gsc = R.DeviceScene(c1, R.BuiltinDesc(9))
        adaptive(gsc, 0.05, 4, 4, 16, 13)
        gsc.close()
        after = plain(c1)
    finally:
        c1.close()
    c2 = R.Context(0)
    try:
        fresh = plain(c2)
    finally:
        c2.close()
    assert after == fresh


@pytest.mark.gpu
def test_tonemap_of_an_adaptive_frame(ctx):
    from tests.test_gpu_render_paths import tonemap_reference
    c = prefix_case(ctx, 7)
    import torch
    acc = c["acc"].astype(np.float32)
    got = c["gsc"].tonemap(torch.from_numpy(acc).cuda()).reshape(-1, 4)
    ref, near = tonemap_reference(acc.reshape(-1, 4))
    diff = got[:, :3].astype(int) - ref.astype(int)
    assert not ((diff != 0) & ~near).any() and (np.abs(diff) <= 1).all() and (got[:, 3] == 255).all()


# ---------------------------------------------------------------------------
# 9: layouts and the CLI
# ---------------------------------------------------------------------------
def test_adaptive_struct_layouts_header_ctypes_and_rust_agree(tmp_path):
    from tests.test_host_cpu import _rust_layout
    ffi = open(os.path.join(ROOT, "rust", "rttnw-b200-sys", "src", "ffi.rs")).read()
    structs = {"rtx_adaptive_params": (abi.AdaptiveParams, 16), "rtx_adaptive_stats": (abi.AdaptiveStats, 24)}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "rttnw_b200.h"', 'int main(void) {']
    for cname, (ct, _) in structs.items():
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in ct._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    c_layout = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, (ct, size) in structs.items():
        rsize, rfields = _rust_layout(ffi, cname)
        assert int(c_layout[cname]) == C.sizeof(ct) == rsize == size
        assert [f for f, _ in ct._fields_] == list(rfields)
        for fname, _ in ct._fields_:
            assert int(c_layout[f"{cname}.{fname}"]) == getattr(ct, fname).offset == rfields[fname]


CLI = os.path.join(ROOT, "rttnw_b200", "lib", "rttnw")


@pytest.mark.parametrize("extra", [["--gpus", "2"], ["--checkpoint", "ck"], ["--resume", "ck"]])
def test_cli_refuses_adaptive_with_several_gpus_or_checkpoints(extra, tmp_path):
    r = subprocess.run([CLI, "7", "--adaptive", "0.01", "--spp", "64"] + extra, cwd=tmp_path, capture_output=True, text=True,
                       timeout=60)
    assert r.returncode == 1 and "--adaptive" in r.stderr and "cannot be combined" in r.stderr
    assert not (tmp_path / "image.png").exists() and "Scene number" not in r.stdout


@pytest.mark.gpu
def test_cli_renders_adaptively(tmp_path):
    r = subprocess.run([CLI, "7", "--adaptive", "0.05", "--spp", "64", "--width", str(W), "--height", str(H)], cwd=tmp_path,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert "Adaptive sampling:" in r.stdout and "tiles converged" in r.stdout
    img = R.png_read_rgba8(str(tmp_path / "image.png"))
    assert img.shape == (H, W, 4) and (img[..., 3] == 255).all() and img[..., :3].mean() > 5
    py = R.render(7, W, H, 64, noise_threshold=0.05)
    assert py.shape == img.shape and np.abs(py.astype(int) - img.astype(int)).mean() < 2.0
