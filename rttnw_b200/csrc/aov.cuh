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

// kEnv (a scene with an environment map): a miss's albedo is env_lookup(env, d) clamped to [0, 1], the background's
// rule applied to the map.
__global__ void __launch_bounds__(kAovBlock) aov_kernel(AovArgs a) {
    constexpr bool kEnv = false;
    const EnvArgs env{};  // (read only when kEnv)
#include "aov_body.cuh"
}

__global__ void __launch_bounds__(kAovBlock) aov_env_kernel(AovArgs a, EnvArgs env) {
    constexpr bool kEnv = true;
#include "aov_body.cuh"
}

}  // namespace rtx
