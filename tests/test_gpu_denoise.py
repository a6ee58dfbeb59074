"""The denoiser (rtx_denoise): the kernels against a float64 restatement of the filter written in rttnw_b200.h,
properties on synthetic frames, refusals, the split render it needs, its quality, and the front ends.

Tolerance of the restatement. The GPU computes in fp32 (unit roundoff u = 2^-24) what denoise_ref computes in f64 from
the same fp32 inputs:
  * the prepass divides at most three times per value (c / n / a', the halves' means, (H - R) / a'), so e carries
    <= 3u relative error and v, a square of a difference of means, <= 16u relative error of the terms it is made of;
  * a weight's exponent x (about ten operations, the reciprocals 1 / sigma^2 rounded once) is off by <= 12u |x|, and
    expf adds 2 ulp, so w is off by a factor 1 + (12 |x| + 2) u; since a tap's share of the mean falls like e^-x, the
    error it causes in the weighted mean is at most max(x e^-x) (12 + 2) u <= 6u times the spread of e in the window;
  * the K-fold weighted means add 25 products and one division per pass: <= 27u of |e| per pass, and each pass
    carries the previous one's error forward through both e and the luminance term.
Summed over K passes that is below 60 K u (|out| + spread) ~ 4e-6 K (|out| + spread). The bound used is 5x that,
2e-5 per pass on |ref| + the frame's mean |ref| (the spread of a window is at most a few frame means in these scenes).
The B200 run DESIGN.md §4 quotes measured at most 6.5e-7 per pass over all scenes, sources and settings
(tests/_record.py keeps it under "denoise"). The inputs are renders, whose atomic sums differ in the last bits from run
to run, so the figure moves a little between runs.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rttnw_b200 as R
from rttnw_b200 import abi
from rttnw_b200.render import DENOISE_DEFAULTS
from tests._record import record
from tests.test_gpu_aov import read_pfm
from tests.test_host_cpu import _rust_layout

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "rttnw_b200", "lib", "rttnw")
LUM = np.array([0.2126, 0.7152, 0.0722])
H5 = np.array([1.0, 4.0, 6.0, 4.0, 1.0]) / 16.0
DEFAULTS = dict(DENOISE_DEFAULTS)
OTHER = {"iterations": 3, "sigma_normal": 0.5, "sigma_albedo": 0.3, "sigma_luminance": 1.5}
RTOL_PASS = 2e-5  # per pass, on |ref| + mean |ref| (module docstring)
# Quality: the denoised frame's display RMSE against a 4096-spp reference is at most F x the raw frame's. The first B200
# run measured 0.305 (scene 7, 16 spp) and 0.447 (scene 9, 64 spp) at sigma_luminance 4, the run at the chosen default
# sigma_luminance 8 0.231 and 0.413; F leaves a third of margin over the first run.
QUALITY_F = {7: 0.45, 9: 0.6}


@pytest.fixture(scope="module")
def ctx():
    c = R.Context(0)
    yield c
    c.close()


# ---------------------------------------------------------------------------
# the float64 restatement (include/rttnw_b200.h, rtx_denoise)
# ---------------------------------------------------------------------------
def _shift(x, dy, dx):
    """x[y + dy, x + dx] where in the frame, 0 elsewhere; and the in-frame mask."""
    h, w = x.shape[:2]
    out = np.zeros_like(x)
    mask = np.zeros((h, w), dtype=bool)
    y0, y1 = max(0, -dy), min(h, h - dy)
    x0, x1 = max(0, -dx), min(w, w - dx)
    if y0 < y1 and x0 < x1:
        out[y0:y1, x0:x1] = x[y0 + dy:y1 + dy, x0 + dx:x1 + dx]
        mask[y0:y1, x0:x1] = True
    return out, mask


def denoise_ref(acc, half, alb, nrm, iterations=5, sigma_normal=0.25, sigma_albedo=0.1, sigma_luminance=8.0):
    acc, half, alb, nrm = (np.asarray(b, dtype=np.float64) for b in (acc, half, alb, nrm))
    n, m = acc[..., 3], half[..., 3]
    valid = n != 0
    with np.errstate(divide="ignore", invalid="ignore"):
        a = np.where(alb[..., 3:4] != 0, alb[..., :3] / alb[..., 3:4], 0.0)
        N = np.where(nrm[..., 3:4] != 0, nrm[..., :3] / nrm[..., 3:4], 0.0)
        ap = np.maximum(a, 1e-3)
        e = np.where(valid[..., None], acc[..., :3] / n[..., None] / ap, 0.0)
        hm = half[..., :3] / m[..., None]
        rm = (acc[..., :3] - half[..., :3]) / (n - m)[..., None]
        v = np.where((m > 0) & (m < n), (((hm - rm) / ap) @ LUM) ** 2 * m * (n - m) / n ** 2, 0.0)
    v = np.where(valid, v, 0.0)
    e = np.where(valid[..., None], e, 0.0)
    feat = np.concatenate([N, a], axis=-1)
    for i in range(iterations):
        s = 2 ** i
        gs, gw = np.zeros_like(v), np.zeros_like(v)
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                vq, inside = _shift(v, dy, dx)
                ok, _ = _shift(valid, dy, dx)
                k = (0.5 if dy == 0 else 0.25) * (0.5 if dx == 0 else 0.25) * (inside & ok)
                gs += k * vq
                gw += k
        with np.errstate(divide="ignore", invalid="ignore"):
            inv_l = 1.0 / (sigma_luminance * np.sqrt(gs / gw) + 1e-10)
        lp = e @ LUM
        sw, se, sv = np.zeros_like(v), np.zeros_like(e), np.zeros_like(v)
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                eq, inside = _shift(e, s * dy, s * dx)
                vq, _ = _shift(v, s * dy, s * dx)
                fq, _ = _shift(feat, s * dy, s * dx)
                ok, _ = _shift(valid, s * dy, s * dx)
                dn = ((feat[..., :3] - fq[..., :3]) ** 2).sum(-1) / sigma_normal ** 2
                da = ((feat[..., 3:] - fq[..., 3:]) ** 2).sum(-1) / sigma_albedo ** 2
                with np.errstate(invalid="ignore", over="ignore"):
                    x = dn + da + np.abs(lp - eq @ LUM) * inv_l
                    w = np.where(inside & ok & valid, H5[dy + 2] * H5[dx + 2] * np.exp(-x), 0.0)
                sw += w
                se += w[..., None] * eq
                sv += w * w * vq
        with np.errstate(divide="ignore", invalid="ignore"):
            e = np.where(valid[..., None], se / sw[..., None], 0.0)
            v = np.where(valid, sv / sw ** 2, 0.0)
    out = np.ones(acc.shape)
    out[..., :3] = np.where(valid[..., None], e * ap, 0.0)
    return out


# ---------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------
def dev(ctx, x):
    t = ctx.torch
    return t.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(f"cuda:{ctx.device}")


def run(ctx, acc, half, alb, nrm, **kw):
    """numpy inputs -> (H, W, 4) float32 numpy output of Context.denoise."""
    out = ctx.denoise(dev(ctx, acc), dev(ctx, half), {"albedo": dev(ctx, alb), "normal": dev(ctx, nrm)}, **kw)
    return out.cpu().numpy()


def check_ref(got, ref, iterations, key=None):
    assert (got[..., 3] == 1).all()
    scale = np.abs(ref[..., :3]).mean()
    ratio = float((np.abs(got[..., :3] - ref[..., :3]) / (np.abs(ref[..., :3]) + scale + 1e-30)).max() / iterations)
    if key:
        record("denoise", key, {"max_error_per_pass": ratio, "allowed": RTOL_PASS})
    assert ratio <= RTOL_PASS, ratio


def display(x):
    """The tonemap of rtx_tonemap_rgba8 before the floor: 8-bit display units."""
    return np.clip(np.sqrt(np.maximum(x, 0.0)), 0.0, 0.999) * 256.0


def synthetic(h, w, rng, n=16, m=8):
    acc = np.zeros((h, w, 4), np.float32)
    col = rng.uniform(0.05, 2.0, (h, w, 3))
    acc[..., :3] = col * n
    acc[..., 3] = n
    half = np.zeros_like(acc)
    half[..., :3] = col * m + rng.normal(0.0, 0.2, (h, w, 3)) * m
    half[..., 3] = m
    alb = np.concatenate([rng.uniform(0.0, 1.0, (h, w, 3)) * 4, np.full((h, w, 1), 4.0)], -1).astype(np.float32)
    nv = rng.normal(size=(h, w, 3))
    nv /= np.linalg.norm(nv, axis=-1, keepdims=True)
    nrm = np.concatenate([nv * 4, np.full((h, w, 1), 4.0)], -1).astype(np.float32)
    return acc, half, alb, nrm


# ---------------------------------------------------------------------------
# 1. real buffers against the restatement
# ---------------------------------------------------------------------------
SCENES = (1, 3, 7, 8, 9)


@pytest.fixture(scope="module")
def real_buffers(ctx):
    """Per scene at 96x96: 16-spp beauty split at 8 (uniform) and adaptive (aux), 8-spp features."""
    out = {}
    for number in SCENES:
        gsc = R.DeviceScene(ctx, R.BuiltinDesc(number))
        w = h = 96
        acc = gsc.new_accum(w, h)
        gsc.render_into(acc, 0, 8, seed=11)
        half = acc.clone()
        gsc.render_into(acc, 8, 8, seed=11)
        acc_a, aux = gsc.new_accum(w, h), gsc.new_accum(w, h)
        gsc.render_adaptive(acc_a, aux, 0.05, 4, 4, 16, seed=11)
        aov = gsc.new_aov(w, h)
        gsc.render_aov(aov, 0, 8, seed=11)
        out[number] = {"uniform": (acc, half), "adaptive": (acc_a, aux), "aov": aov}
        gsc.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("number", SCENES)
@pytest.mark.parametrize("source", ["uniform", "adaptive"])
def test_real_buffers_match_the_float64_restatement(ctx, real_buffers, number, source):
    b = real_buffers[number]
    acc, half = b[source]
    np_in = [x.cpu().numpy() for x in (acc, half, b["aov"]["albedo"], b["aov"]["normal"])]
    if source == "uniform":
        assert (np_in[1][..., 3] == 8).all() and (np_in[0][..., 3] == 16).all()
    else:
        assert (np_in[1][..., 3] * 2 == np_in[0][..., 3]).all()
    for params in (DEFAULTS, OTHER):
        for k in (1, 5):
            p = dict(params, iterations=k)
            got = ctx.denoise(acc, half, b["aov"], **p).cpu().numpy()
            ref = denoise_ref(*np_in, **p)
            check_ref(got, ref, k, key=f"scene{number}_{source}_K{k}_{'default' if params is DEFAULTS else 'other'}")


# ---------------------------------------------------------------------------
# 2. properties on synthetic frames
# ---------------------------------------------------------------------------
@pytest.mark.gpu
def test_constant_frame_stays_constant(ctx):
    h, w = 40, 56
    acc = np.zeros((h, w, 4), np.float32)
    acc[...] = (0.3 * 16, 0.6 * 16, 1.2 * 16, 16)
    half = acc * 0.5
    alb = np.broadcast_to(np.float32([0.4, 0.5, 0.6, 1.0]), (h, w, 4))
    nrm = np.broadcast_to(np.float32([0.0, 0.0, 1.0, 1.0]), (h, w, 4))
    out = run(ctx, acc, half, alb, nrm)
    assert np.allclose(out[..., :3], [0.3, 0.6, 1.2], rtol=1e-6, atol=0) and (out[..., 3] == 1).all()


@pytest.mark.gpu
def test_zero_variance_frame_comes_back_unchanged(ctx):
    rng = np.random.default_rng(1)
    acc, _, alb, nrm = synthetic(48, 64, rng)
    half = acc.copy()
    half[..., :3] *= 0.5  # half = accum * m / n, exact in fp32
    half[..., 3] = 8
    out = run(ctx, acc, half, alb, nrm)
    c = acc[..., :3].astype(np.float64) / 16
    assert (np.abs(out[..., :3] - c) <= 8 * 2.0 ** -24 * c).all()


def step_frame(kind, rng, h=32, w=32, delta=0.0):
    """Left half | right half. 'normal': orthogonal normals, same albedo; 'miss': a surface against a miss (normal 0,
    another albedo). delta (a power of two) is added to the right side's mean colour. Colours and noise lie on a 2^-8
    grid, so the sums, the halves' means and H - R are exact in fp32 and v is bit for bit the same."""
    _, _, alb, nrm = synthetic(h, w, rng)
    col = np.round(rng.uniform(0.05, 2.0, (h, w, 3)) * 256) / 256
    noise = np.round(rng.normal(0.0, 0.2, (h, w, 3)) * 256) / 256
    acc = np.concatenate([col * 16, np.full((h, w, 1), 16.0)], -1).astype(np.float32)
    half = np.concatenate([(col + noise) * 8, np.full((h, w, 1), 8.0)], -1).astype(np.float32)
    alb[..., :3] = 0.5 * 4
    nrm[..., :w // 2, :3] = (4.0, 0.0, 0.0)
    if kind == "normal":
        nrm[..., w // 2:, :3] = (0.0, 4.0, 0.0)
    else:
        nrm[..., w // 2:, :3] = 0.0
        alb[..., w // 2:, :3] = 0.8 * 4
    acc[:, w // 2:, :3] += delta * 16
    half[:, w // 2:, :3] += delta * 8
    return acc, half, alb, nrm


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["normal", "miss"])
def test_perturbing_one_side_of_an_edge_barely_moves_the_other(ctx, kind):
    """One pass: its variance input v is the same bit for bit, so the near side's own weights do not change and the far
    side moves it through the cross-edge taps alone. (Over several passes the 3x3 blur g of v, which is not
    edge-aware, also carries the far side's rounding across the edge.)"""
    h, w, delta = 32, 32, 64.0
    base = run(ctx, *step_frame(kind, np.random.default_rng(2)), iterations=1)
    moved = run(ctx, *step_frame(kind, np.random.default_rng(2), delta=delta), iterations=1)
    # a tap across the edge has exp(-x) times the weight it would have, x >= |dN|^2 / sn^2 + |da|^2 / sa^2; the
    # non-centre taps hold 1 - (6/16)^2 of the kernel against (6/16)^2 for the centre, so the far side holds at most a
    # share q of the weight and moves the near side by at most q (delta / a' + spread) a', plus the rounding of the sums
    x = (2.0 if kind == "normal" else 1.0) / 0.25 ** 2 + (0.0 if kind == "normal" else 3 * 0.3 ** 2 / 0.1 ** 2)
    q = np.exp(-x) * (1 - (6 / 16) ** 2) / (6 / 16) ** 2
    spread = base[..., :3].max() / 0.5
    bound = q * (delta / 0.5 + spread) * 0.5 + 8 * 2.0 ** -24 * np.abs(base[:, :w // 2, :3])
    assert (np.abs(moved[:, :w // 2, :3] - base[:, :w // 2, :3]) <= bound).all()
    assert (np.abs(moved[:, w // 2:, :3] - base[:, w // 2:, :3]) > delta / 2).all()  # the far side did move


@pytest.mark.gpu
def test_pixels_without_samples_output_zero_and_contribute_nothing(ctx):
    rng = np.random.default_rng(3)
    acc, half, alb, nrm = synthetic(40, 40, rng)
    holes = rng.uniform(size=(40, 40)) < 0.2
    acc[holes] = 0.0
    half[holes] = 0.0
    out = run(ctx, acc, half, alb, nrm)
    assert (out[holes] == [0, 0, 0, 1]).all()
    check_ref(out, denoise_ref(acc, half, alb, nrm), 5)
    # whatever sits in the colour, half and feature buffers of a pixel with n == 0 changes nothing
    acc2, half2, alb2, nrm2 = acc.copy(), half.copy(), alb.copy(), nrm.copy()
    acc2[holes, :3] = 1e30
    half2[holes] = (5.0, -5.0, 1e20, 3.0)
    alb2[holes] = (9.0, 0.0, 3.0, 1.0)
    nrm2[holes] = (-1.0, 7.0, 0.0, 1.0)
    assert np.array_equal(run(ctx, acc2, half2, alb2, nrm2), out)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1, 1), (3, 7), (17, 33), (1, 800)])
def test_small_and_thin_frames_with_steps_wider_than_the_frame(ctx, shape):
    h, w = shape
    rng = np.random.default_rng(h * 1000 + w)
    acc, half, alb, nrm = synthetic(h, w, rng)
    for k in (1, 10):
        check_ref(run(ctx, acc, half, alb, nrm, iterations=k), denoise_ref(acc, half, alb, nrm, iterations=k), k)


@pytest.mark.gpu
def test_tiny_sigmas_give_a_finite_frame(ctx):
    """The smallest accepted sigma_normal / sigma_albedo (1 / sigma^2 just below the fp32 maximum) and a tiny
    sigma_luminance leave every tap but the centre at weight 0: the frame comes back as it went in, finite."""
    rng = np.random.default_rng(6)
    acc, half, alb, nrm = synthetic(24, 40, rng)
    for s in ({"sigma_normal": 1e-19}, {"sigma_albedo": 1e-19}, {"sigma_luminance": 1e-30}):
        out = run(ctx, acc, half, alb, nrm, **s)
        assert np.isfinite(out).all(), s
        check_ref(out, denoise_ref(acc, half, alb, nrm, **dict(DEFAULTS, **s)), 5)


@pytest.mark.gpu
def test_frame_taller_than_a_2d_grid_allows(ctx):
    """600 000 rows: more than 65 535 rows of 8-pixel-high blocks, which a 2D launch could not cover."""
    rng = np.random.default_rng(7)
    acc, half, alb, nrm = synthetic(600000, 2, rng)
    check_ref(run(ctx, acc, half, alb, nrm, iterations=2), denoise_ref(acc, half, alb, nrm, iterations=2), 2)


@pytest.mark.gpu
def test_deterministic_and_inputs_unchanged(ctx):
    rng = np.random.default_rng(4)
    bufs = [dev(ctx, x) for x in synthetic(64, 96, rng)]
    before = [b.clone() for b in bufs]
    aov = {"albedo": bufs[2], "normal": bufs[3]}
    a = ctx.denoise(bufs[0], bufs[1], aov)
    b = ctx.denoise(bufs[0], bufs[1], aov)
    assert ctx.torch.equal(a, b)
    c = ctx.torch.empty_like(a)  # params == NULL: the defaults
    abi.check(ctx.lib.rtx_denoise(ctx.h, *(x.data_ptr() for x in bufs), 96, 64, None, c.data_ptr()))
    assert ctx.torch.equal(a, c)
    for x, y in zip(bufs, before):
        assert ctx.torch.equal(x, y)


# ---------------------------------------------------------------------------
# 3. refusals and rtx_memcpy_d2d
# ---------------------------------------------------------------------------
@pytest.mark.gpu
def test_refusals(ctx):
    lib = ctx.lib
    t = ctx.torch
    w, h = 16, 8
    bufs = [t.zeros((h, w, 4), dtype=t.float32, device="cuda:0") for _ in range(5)]
    ptrs = [b.data_ptr() for b in bufs]

    def call(p=None, ww=w, hh=h, ptr=None, params=abi.DenoiseParams(5, 0.25, 0.1, 4.0)):
        p = list(ptrs) if p is None else p
        return lib.rtx_denoise(ctx.h, p[0], p[1], p[2], p[3], ww, hh, C.byref(params) if params else None,
                               p[4] if ptr is None else ptr)

    assert call() == abi.RTX_OK and call(params=None) == abi.RTX_OK
    assert lib.rtx_denoise(None, *ptrs[:4], w, h, None, ptrs[4]) == -1
    for i in range(5):
        p = list(ptrs)
        p[i] = None
        assert call(p) == -1, i
    for ww, hh in ((0, 8), (16, 0), (-1, 8), (16, -3), (65536, 32768)):
        assert call(ww=ww, hh=hh) == -1, (ww, hh)
    for it in (0, 11, -1):
        assert call(params=abi.DenoiseParams(it, 0.25, 0.1, 4.0)) == -1, it
    for bad in (0.0, -1.0, float("inf"), float("nan")):
        for j in range(3):
            s = [0.25, 0.1, 4.0]
            s[j] = bad
            assert call(params=abi.DenoiseParams(5, *s)) == -1, (bad, j)
    n = w * h * 16
    for i in range(4):
        assert call(ptr=ptrs[i]) == -1
        assert call(ptr=ptrs[i] + n - 16) == -1  # the output's first float4 is the input's last
        assert call(ptr=ptrs[i] - n + 16) == -1  # the output's last float4 is the input's first
    big = t.zeros((4, h, w, 4), dtype=t.float32, device="cuda:0")
    assert call(ptr=big.data_ptr()) == abi.RTX_OK
    # every buffer must be float4-aligned: misaligned pointers are refused, not faulted on
    for off in (4, 8, 12):
        assert call(ptr=big.data_ptr() + off) == -1, off
        for i in range(4):
            p = list(ptrs)
            p[i] = big.data_ptr() + n * 2 + off  # inside `big`, clear of d_out
            assert call(p) == -1, (i, off)
    # 1 / sigma^2 must be finite in fp32 for sigma_normal and sigma_albedo (about 5.4e-20 and up)
    for j in range(2):
        s = [0.25, 0.1, 8.0]
        s[j] = 1e-20
        assert call(params=abi.DenoiseParams(5, *s)) == -1, j
    ctx.sync()


@pytest.mark.gpu
def test_memcpy_d2d_round_trip_and_refusal(ctx):
    t = ctx.torch
    src = t.arange(1000, dtype=t.float32, device="cuda:0")
    dst = t.zeros_like(src)
    abi.check(ctx.lib.rtx_memcpy_d2d(ctx.h, dst.data_ptr(), src.data_ptr(), 4000))
    back = t.zeros_like(src)
    abi.check(ctx.lib.rtx_memcpy_d2d(ctx.h, back.data_ptr(), dst.data_ptr(), 4000))
    ctx.sync()
    assert t.equal(back, src)
    assert ctx.lib.rtx_memcpy_d2d(ctx.h, None, src.data_ptr(), 4) == -1
    assert ctx.lib.rtx_memcpy_d2d(ctx.h, dst.data_ptr(), None, 4) == -1
    assert ctx.lib.rtx_memcpy_d2d(None, dst.data_ptr(), src.data_ptr(), 4) == -1


# ---------------------------------------------------------------------------
# 4. the split render, and quality
# ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("number", [7, 9])
def test_render_split_at_half_equals_one_render(ctx, number):
    """The sums differ only in fp32 summation order: each is within (n - 1) u of the exact sum of non-negative terms."""
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(number))
    one = gsc.new_accum(64, 48)
    gsc.render_into(one, 0, 32, seed=5)
    two = gsc.new_accum(64, 48)
    gsc.render_into(two, 0, 16, seed=5)
    half = two.clone()
    gsc.render_into(two, 16, 16, seed=5)
    a, b = one.cpu().numpy().astype(np.float64), two.cpu().numpy().astype(np.float64)
    assert (a[..., 3] == 32).all() and (b[..., 3] == 32).all() and (half.cpu().numpy()[..., 3] == 16).all()
    assert (np.abs(a[..., :3] - b[..., :3]) <= 2 * 32 * 2.0 ** -24 * np.maximum(a[..., :3], b[..., :3]) + 1e-30).all()
    gsc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("number,spp", [(7, 16), (9, 64)])
def test_denoised_frame_is_closer_to_the_reference(ctx, number, spp):
    w = h = 128
    gsc = R.DeviceScene(ctx, R.BuiltinDesc(number))
    ref = gsc.new_accum(w, h)
    gsc.render_into(ref, 1 << 20, 4096, seed=3)  # sample indices disjoint from the frame's
    acc = gsc.new_accum(w, h)
    gsc.render_into(acc, 0, spp // 2, seed=3)
    half = acc.clone()
    gsc.render_into(acc, spp // 2, spp - spp // 2, seed=3)
    aov = gsc.new_aov(w, h)
    gsc.render_aov(aov, 0, min(16, spp), seed=3)
    den = ctx.denoise(acc, half, aov).cpu().numpy().astype(np.float64)
    r = ref.cpu().numpy().astype(np.float64)
    a = acc.cpu().numpy().astype(np.float64)
    want = display(r[..., :3] / r[..., 3:])
    raw = np.sqrt(np.mean((display(a[..., :3] / a[..., 3:]) - want) ** 2))
    out = np.sqrt(np.mean((display(den[..., :3]) - want) ** 2))
    record("denoise", f"quality_scene{number}_{spp}spp", {"raw_rmse": raw, "denoised_rmse": out, "ratio": out / raw,
                                                          "allowed": QUALITY_F[number]})
    assert out <= QUALITY_F[number] * raw, (out, raw)
    gsc.close()


# ---------------------------------------------------------------------------
# 5. front ends
# ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("threshold", [None, 0.05])
def test_python_render_denoise_is_the_tonemap_of_context_denoise(tmp_path, monkeypatch, threshold):
    seen = {}
    orig = R.Context.denoise

    def spy(self, accum, half, aov, **kw):
        out = orig(self, accum, half, aov, **kw)
        rgba = np.zeros(out.shape[:2] + (4,), np.uint8)
        abi.check(self.lib.rtx_tonemap_rgba8(self.h, out.data_ptr(), out.shape[1], out.shape[0], rgba.ctypes.data, 0))
        seen.update(rgba=rgba, n=accum[..., 3].cpu().numpy(), m=half[..., 3].cpu().numpy(),
                    feat=aov["albedo"][..., 3].cpu().numpy(), out=out.cpu().numpy())
        return out

    monkeypatch.setattr(R.Context, "denoise", spy)
    w, h = 48, 32
    png = str(tmp_path / "image.png")
    rgba = R.render(7, w, h, 16, out_path=png, noise_threshold=threshold, aov_prefix=str(tmp_path / "out"),
                    aov_samples=4, denoise=True)
    assert np.array_equal(rgba, seen["rgba"]) and np.array_equal(R.png_read_rgba8(png), rgba)
    assert (seen["feat"] == 4).all()
    if threshold is None:
        assert (seen["n"] == 16).all() and (seen["m"] == 8).all()
    else:
        assert (seen["m"] * 2 == seen["n"]).all()
    assert np.array_equal(read_pfm(tmp_path / "out.denoised.pfm"), seen["out"][..., :3])


def tonemap_np(x):
    return np.floor(np.clip(np.sqrt(x.astype(np.float64)), 0.0, 0.999) * 256.0)


@pytest.mark.gpu
@pytest.mark.parametrize("extra,w,h", [(["--aov-spp", "4"], 64, 48), (["--aov", "out"], 64, 48),
                                       (["--adaptive", "0.05"], 64, 48), (["--adaptive", "0.05", "--aov", "out"], 64, 48),
                                       (["--aov-spp", "4"], 63, 47), (["--aov", "out"], 63, 47),
                                       (["--adaptive", "0.05", "--aov", "out"], 63, 47)])
def test_cli_denoise(extra, w, h, tmp_path):
    """Uniform and adaptive paths, with and without the PFMs; 63x47 has an odd pixel count, so a buffer carved out of
    the feature block behind the float2 depth would not be float4-aligned."""
    r = subprocess.run([CLI, "7", "--width", str(w), "--height", str(h), "--spp", "16", "--denoise"] + extra,
                       cwd=tmp_path, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    img = R.png_read_rgba8(str(tmp_path / "image.png"))
    assert img.shape == (h, w, 4)
    if "--aov" in extra:
        den = read_pfm(tmp_path / "out.denoised.pfm")
        beauty = read_pfm(tmp_path / "out.beauty.pfm")
        assert (np.abs(tonemap_np(den) - img[..., :3]) <= 1).all()  # image.png is the denoised frame
        assert not np.array_equal(den, beauty)
    else:
        assert sorted(os.listdir(tmp_path)) == ["image.png"]


@pytest.mark.parametrize("args", [["--gpus", "2"], ["--checkpoint", "ck"], ["--resume", "ck"]])
def test_cli_refuses_denoise_with_several_gpus_or_checkpoints(args, tmp_path):
    r = subprocess.run([CLI, "7", "--spp", "8", "--denoise"] + args, cwd=tmp_path, capture_output=True, text=True,
                       timeout=60)
    assert r.returncode == 1 and "--denoise" in r.stderr
    assert "Scene number" not in r.stdout and not list(tmp_path.iterdir())


def test_denoise_params_layout_header_ctypes_and_rust_agree(tmp_path):
    src = tmp_path / "layout.c"
    fields = [f for f, _ in abi.DenoiseParams._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "rttnw_b200.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(rtx_denoise_params));']
    lines += [f'  printf("{f} %zu\\n", offsetof(rtx_denoise_params, {f}));' for f in fields]
    lines += ['  return 0;', '}']
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    c_layout = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True,
                                                      text=True).stdout.splitlines())
    ffi = open(os.path.join(ROOT, "rust", "rttnw-b200-sys", "src", "ffi.rs")).read()
    rsize, rfields = _rust_layout(ffi, "rtx_denoise_params")
    assert int(c_layout["size"]) == C.sizeof(abi.DenoiseParams) == rsize == 16
    assert list(rfields) == fields
    for f in fields:
        assert int(c_layout[f]) == getattr(abi.DenoiseParams, f).offset == rfields[f]


def test_defaults_agree_between_python_and_rust():
    ffi = open(os.path.join(ROOT, "rust", "rttnw-b200-sys", "src", "ffi.rs")).read()
    d = DEFAULTS
    assert (f"iterations: {d['iterations']}, sigma_normal: {d['sigma_normal']}, sigma_albedo: {d['sigma_albedo']}, "
            f"sigma_luminance: {d['sigma_luminance']}") in ffi
