// denoise.cuh — the feature-guided à-trous filter of rtx_denoise (the exact filter is written out in rttnw_b200.h).
//
// Shape: a prepass turns the caller's four float4 buffers into per-pixel scratch the taps read: the static features
// {N.xyz, a.r} (16 B) and {a.g, a.b} (8 B), and the filtered quantity {e.rgb, v} (16 B; v < 0 marks a pixel without
// samples, a valid v is >= 0). Then one à-trous kernel runs once per pass with step 2^i, ping-ponging {e, v} between
// two scratch buffers; the last pass remodulates into the caller's output instead. One thread per pixel over 32x8
// tiles, numbered along a 1D grid (a 2D grid's 65 535 rows of blocks would cap the height), taps summed in a fixed order in registers: no atomics, bit-identical from run to run. Each tap reads 40 B;
// the whole working set (56 B per pixel, 36 MB at 800x800) stays in L2, and shared-memory staging was not built
// (DESIGN.md §4 has the measured time).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace rtx {

constexpr int kDenoiseBX = 32, kDenoiseBY = 8;

// The pixel of this thread: block b is tile (b % tiles_x, b / tiles_x). 64-bit, as are the tap coordinates: a frame
// may be up to 2^31 - 1 pixels wide, and x + 2^9 * 2 would overflow an int there.
__device__ __forceinline__ void dn_pixel(int tiles_x, int64_t& x, int64_t& y) {
    const int64_t ty = blockIdx.x / (unsigned)tiles_x, tx = blockIdx.x - ty * tiles_x;
    x = tx * kDenoiseBX + threadIdx.x;
    y = ty * kDenoiseBY + threadIdx.y;
}

// Explicitly rounded so that the compiler cannot contract it differently at different call sites: the centre tap's
// |L(e_p) - L(e_q)| must be exactly 0, or where g_p = 0 (1e10 / sigma_l per unit of luminance) even the centre weight
// underflows and sum w = 0.
__device__ __forceinline__ float dn_lum(float r, float g, float b) {
    return __fmaf_rn(0.0722f, b, __fmaf_rn(0.7152f, g, __fmul_rn(0.2126f, r)));
}

__global__ void __launch_bounds__(kDenoiseBX * kDenoiseBY)
denoise_prepass_kernel(const float4* __restrict__ accum, const float4* __restrict__ half, const float4* __restrict__ albedo,
                       const float4* __restrict__ normal, int width, int height, int tiles_x, float4* __restrict__ feat0,
                       float2* __restrict__ feat1, float4* __restrict__ ev) {
    int64_t x, y;
    dn_pixel(tiles_x, x, y);
    if (x >= width || y >= height) return;
    const size_t p = (size_t)(y * width + x);
    const float4 c = accum[p], h = half[p], al = albedo[p], nm = normal[p];
    float ar = 0.f, ag = 0.f, ab = 0.f, nx = 0.f, ny = 0.f, nz = 0.f;
    if (al.w != 0.f) { ar = al.x / al.w; ag = al.y / al.w; ab = al.z / al.w; }
    if (nm.w != 0.f) { nx = nm.x / nm.w; ny = nm.y / nm.w; nz = nm.z / nm.w; }
    feat0[p] = make_float4(nx, ny, nz, ar);
    feat1[p] = make_float2(ag, ab);
    const float n = c.w, m = h.w;
    if (!(n != 0.f)) {  // no samples: contributes nothing, outputs {0, 0, 0, 1}
        ev[p] = make_float4(0.f, 0.f, 0.f, -1.f);
        return;
    }
    const float qr = fmaxf(ar, 1e-3f), qg = fmaxf(ag, 1e-3f), qb = fmaxf(ab, 1e-3f);  // a'
    const float er = c.x / n / qr, eg = c.y / n / qg, eb = c.z / n / qb;
    float v = 0.f;
    if (m > 0.f && m < n) {
        const float k = n - m;
        const float dr = (h.x / m - (c.x - h.x) / k) / qr, dg = (h.y / m - (c.y - h.y) / k) / qg,
                    db = (h.z / m - (c.z - h.z) / k) / qb;
        const float l = dn_lum(dr, dg, db);
        v = l * l * ((m / n) * (k / n));
    }
    ev[p] = make_float4(er, eg, eb, v);
}

struct DenoisePass {
    const float4* feat0;
    const float2* feat1;
    const float4* ev_in;
    float4* ev_out;  // passes 0 .. K-2
    float4* out;     // the last pass: {e * a', 1}
    int width, height, tiles_x, step;
    float inv_sn2, inv_sa2, sigma_l;  // 1 / sigma_n^2, 1 / sigma_a^2, sigma_l
};

__global__ void __launch_bounds__(kDenoiseBX * kDenoiseBY) denoise_atrous_kernel(DenoisePass a) {
    int64_t x, y;
    dn_pixel(a.tiles_x, x, y);
    if (x >= a.width || y >= a.height) return;
    const size_t p = (size_t)(y * a.width + x);
    const float4 cp = a.ev_in[p];
    if (cp.w < 0.f) {
        if (a.out) a.out[p] = make_float4(0.f, 0.f, 0.f, 1.f);
        else a.ev_out[p] = cp;
        return;
    }
    // g_p: the [1/4, 1/2, 1/4]^2 blur of v over in-frame pixels with samples, renormalised
    float gs = 0.f, gw = 0.f;
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy) {
        const int64_t qy = y + dy;
        if (qy < 0 || qy >= a.height) continue;
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
            const int64_t qx = x + dx;
            if (qx < 0 || qx >= a.width) continue;
            const float vq = a.ev_in[(size_t)(qy * a.width + qx)].w;
            if (vq < 0.f) continue;
            const float k = (dy == 0 ? 0.5f : 0.25f) * (dx == 0 ? 0.5f : 0.25f);
            gs += k * vq;
            gw += k;
        }
    }
    const float inv_l = 1.f / (a.sigma_l * sqrtf(gs / gw) + 1e-10f);
    const float4 fp0 = a.feat0[p];
    const float2 fp1 = a.feat1[p];
    const float lp = dn_lum(cp.x, cp.y, cp.z);
    const float hk[5] = {1.f / 16.f, 4.f / 16.f, 6.f / 16.f, 4.f / 16.f, 1.f / 16.f};
    float sw = 0.f, sr = 0.f, sg = 0.f, sb = 0.f, sv = 0.f;
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy) {
        const int64_t qy = y + a.step * dy;
        if (qy < 0 || qy >= a.height) continue;
#pragma unroll
        for (int dx = -2; dx <= 2; ++dx) {
            const int64_t qx = x + a.step * dx;
            if (qx < 0 || qx >= a.width) continue;
            const size_t q = (size_t)(qy * a.width + qx);
            const float4 eq = a.ev_in[q];
            if (eq.w < 0.f) continue;
            const float4 f0 = a.feat0[q];
            const float2 f1 = a.feat1[q];
            const float dnx = fp0.x - f0.x, dny = fp0.y - f0.y, dnz = fp0.z - f0.z;
            const float dar = fp0.w - f0.w, dag = fp1.x - f1.x, dab = fp1.y - f1.y;
            const float dl = fabsf(__fsub_rn(lp, dn_lum(eq.x, eq.y, eq.z)));
            const float w = hk[dy + 2] * hk[dx + 2] *
                            expf(-(dnx * dnx + dny * dny + dnz * dnz) * a.inv_sn2 -
                                 (dar * dar + dag * dag + dab * dab) * a.inv_sa2 - dl * inv_l);
            sw += w;
            sr += w * eq.x; sg += w * eq.y; sb += w * eq.z;
            sv += w * w * eq.w;
        }
    }
    const float er = sr / sw, eg = sg / sw, eb = sb / sw;  // sw >= (6/16)^2: the centre tap has weight h(0)^2
    if (a.out) {
        a.out[p] = make_float4(er * fmaxf(fp0.w, 1e-3f), eg * fmaxf(fp1.x, 1e-3f), eb * fmaxf(fp1.y, 1e-3f), 1.f);
    } else {
        a.ev_out[p] = make_float4(er, eg, eb, sv / (sw * sw));
    }
}

}  // namespace rtx
