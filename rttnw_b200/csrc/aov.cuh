// aov.cuh — the feature-buffer pass (rtx_render_aov): albedo, normal and distance of the first vertex of every path.
//
// Sample s of a pixel gets the buffers of the first vertex of THAT path s of rtx_render with the same seed: the same
// camera ray (camera_ray: jitter, lens, shutter time), the same closest surface hit over the world BVH in [0.001, inf),
// and the same bounce-0 free-flight draw of every ConstantMedium (media_after with the bounce-0 sampler), so the vertex
// is the one wf_shade2_kernel shades at bounce 0, with the same fp32 / f64 split. A denoiser wants the linear beauty
// plus these buffers of the same samples; a compositor wants the distance.
//
// Shape: a warp covers one 8x4 tile, one lane per pixel, and each lane loops over the call's samples in ascending
// order, summing in registers; the sums are added to the buffers once per call. One thread owns a pixel, so there are
// no atomics and the result is bit-identical from run to run.
#pragma once
#include "shade2.cuh"

namespace rtx {

constexpr int kAovBlock = 128;

struct AovArgs {
    SceneView sc;
    CameraView cam;
    int32_t width, height, spp_begin, spp_count;
    uint32_t k0, k1;
    int32_t tiles_x;
    float4* albedo;  // each may be null: not wanted
    float4* normal;
    float2* depth;
};

__global__ void __launch_bounds__(kAovBlock) aov_kernel(AovArgs a) {
    const int warp = (int)((blockIdx.x * (unsigned)kAovBlock + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    const int ty = warp / a.tiles_x, tx = warp - ty * a.tiles_x;
    const int px = tx * kTileW + (lane & (kTileW - 1));
    const int row = ty * kTileH + lane / kTileW;  // row 0 = top
    if (px >= a.width || row >= a.height) return;
    int32_t stack[kStackSize];
    Tally<false> tally;
    const SceneView& sc = a.sc;
    Sampler smp{a.k0, a.k1, (uint32_t)(row * a.width + px), 0u, 0u};
    float al_r = 0.f, al_g = 0.f, al_b = 0.f;
    float n_x = 0.f, n_y = 0.f, n_z = 0.f;
    float dist = 0.f, hits = 0.f;
    const float bg_r = fminf(fmaxf(a.cam.background[0], 0.f), 1.f), bg_g = fminf(fmaxf(a.cam.background[1], 0.f), 1.f),
                bg_b = fminf(fmaxf(a.cam.background[2], 0.f), 1.f);
#pragma unroll 1
    for (int s = 0; s < a.spp_count; ++s) {
        smp.sample = (uint32_t)a.spp_begin + (uint32_t)s;
        RayD ray;
        camera_ray(a.cam, a.width, a.height, px, a.height - 1 - row, smp, ray);
        Best best{1.7976931348623157e308, -1, 0};  // what the shade kernel leaves in the pool for a camera ray
        traverse_simple(sc, sc.world_root, ray, 0.001, best, stack, 0, tally);
        if (sc.n_media > 0) media_after(sc, ray, 0.001, best, smp, stack, tally);
        if (best.rec < 0) {  // background (Q8)
            al_r += bg_r; al_g += bg_g; al_b += bg_b;
            continue;
        }
        HitOut ho;
        finalize_hit<false>(sc, ray, best, ho);
        dist += (float)(best.t * sqrt(dot(ray.d, ray.d)));
        hits += 1.f;
        int32_t mkind, mtex = 0;
        float r = 1.f, g = 1.f, b = 1.f;  // Dielectric: the attenuation (1, 1, 1), material.rs:189
        if (ho.material < 0) {  // ConstantMedium's own Isotropic (hittable.rs:726,786): its normal is arbitrary, count 0
            mkind = RTX_MAT_ISOTROPIC;
            mtex = -(ho.material + 1);
        } else {
            const DMaterial m = sc.materials[ho.material];
            mkind = m.kind;
            mtex = m.texture;
            if (mkind == RTX_MAT_METAL) { r = m.albedo[0]; g = m.albedo[1]; b = m.albedo[2]; }  // absorbed or not
            n_x += (float)ho.n.x; n_y += (float)ho.n.y; n_z += (float)ho.n.z;
        }
        // Texture::value with shade_hit's uv rules (kernels.cuh shade_hit; restated here so that the render kernels keep
        // their code): only image textures look at (u, v), moving spheres and media have u = v = 0
        if (mkind == RTX_MAT_LAMBERTIAN || mkind == RTX_MAT_ISOTROPIC || mkind == RTX_MAT_DIFFUSE_LIGHT) {
            float tu = 0.f, tv = 0.f;
            if (sc.textures[mtex]._pad) {
                if (ho.type == REC_SPHERE) {  // Sphere::uv (hittable.rs:77-83) in fp32
                    const float PI = 3.14159265358979f;
                    tv = acosf(-(float)ho.on.y) / PI;
                    tu = (atan2f(-(float)ho.on.z, (float)ho.on.x) + PI) / (2.f * PI);
                } else if (ho.type >= REC_RECT_XY && ho.type <= REC_RECT_YZ) {
                    rect_uv(sc, best.rec, ho.ru, ho.rv, tu, tv);
                }
            }
            const DTexture t = resolve_texture(sc, mtex, ho.p);
            const f3 tex = texture_eval(sc, t, tu, tv, ho.p);
            r = tex.x; g = tex.y; b = tex.z;
            if (mkind == RTX_MAT_DIFFUSE_LIGHT) {  // emission clamped to the albedo range
                r = fminf(fmaxf(r, 0.f), 1.f); g = fminf(fmaxf(g, 0.f), 1.f); b = fminf(fmaxf(b, 0.f), 1.f);
            }
        }
        al_r += r; al_g += g; al_b += b;
    }
    const size_t pix = smp.pixel;
    const float n = (float)a.spp_count;
    if (a.albedo) {
        float4 v = a.albedo[pix];
        a.albedo[pix] = make_float4(v.x + al_r, v.y + al_g, v.z + al_b, v.w + n);
    }
    if (a.normal) {
        float4 v = a.normal[pix];
        a.normal[pix] = make_float4(v.x + n_x, v.y + n_y, v.z + n_z, v.w + n);
    }
    if (a.depth) {
        float2 v = a.depth[pix];
        a.depth[pix] = make_float2(v.x + dist, v.y + hits);
    }
}

}  // namespace rtx
