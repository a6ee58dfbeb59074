// shade2.cuh — K2a, second form: one level of color() per slot, with the two things the ncu source view of the first
// form (wf_shade_kernel) shows its warps waiting for taken off the critical path, and the work 90 % of the rays threw
// away not done at all.
//
//  * The sample dispenser. The first form read the dispenser ("already dry?") and then did the atomic, two dependent L2
//    round trips at the very end of the warp's critical path (16.7 % of its stall samples, kernels.cuh:1245 and the
//    atomicAdd). Here the read is issued with the first pool load, at the top of the kernel; the atomic still follows
//    the shading, because which lanes ended is only known then. Worth 5 % on the Cornell box (712 -> 752 M samples/s,
//    40 % of whose slots end per pass), 0.5 % on the final scene.
//  * ConstantMedium::hit (hittable.rs:740-796) after the surface search instead of before it. The first form evaluated
//    every medium for every new ray — an f64 quadratic, a square root and a logarithm for the fog that fills the final
//    scene — so that the scatter distance could bound the traversal. But the free-flight distance -ln(u) / density is
//    known from one fp32 logarithm, and once the surface hit is known a ray cannot scatter unless that distance fits
//    into [t_min, t_surface]: for the final scene's fog (mean free path 10^4 against surface distances of 10^2..10^3)
//    that skips the boundary test for every ray that hit a surface nearby: the medium tests per ray fall from 1.35 to
//    0.57 (what is left are the rays that hit nothing, for which the segment is unbounded, and the small medium), while
//    the traversal, no longer cut short by a scatter point, visits 4.5 % more nodes. The closest candidate wins either way, so the answer is
//    the reference's whatever the order (SURVEY.md hard parts); the filter only uses bounds that err on the side of
//    running the exact test.
//
// Same Philox counters, same results as the first form (tests/test_gpu_parity.py::test_other_kernel_forms_trace_the_same_rays).
#pragma once
#include "kernels.cuh"

namespace rtx {

// Every medium that can scatter the ray before best.t. Medium k draws word (k & 3) of Philox block (MEDIUM, k >> 2).
template <bool kCount>
__device__ __forceinline__ void media_after(const SceneView& sc, const RayD& ray, double tmin, Best& best, const Sampler& smp,
                                            int32_t* stack, Tally<kCount>& tally) {
    // upper bound of the length of [tmin, best.t] along the ray, in fp32 (inf when nothing was hit)
    const float dx = (float)ray.d.x, dy = (float)ray.d.y, dz = (float)ray.d.z;
    const float len_ub = sqrtf(fmaf(dx, dx, fmaf(dy, dy, dz * dz))) * 1.000001f;
    const float seg_ub = (__double2float_ru(best.t) - __double2float_rd(tmin)) * len_ub * 1.000001f;
    uint4 w = make_uint4(0, 0, 0, 0);
    int32_t w_block = -1;
    bool have_slab = false;
    SlabRay s;
    for (int32_t m = 0; m < sc.n_media; ++m) {
        const float4* mp = reinterpret_cast<const float4*>(sc.media + m);
        const float4 lo = __ldg(mp), hi = __ldg(mp + 1);
        const float inv_density_lb = __ldg(reinterpret_cast<const float*>(mp + 2));
        const int32_t ord = __float_as_int(hi.w);
        if ((ord >> 2) != w_block) {
            w_block = ord >> 2;
            w = smp.block(P_MEDIUM, (uint32_t)w_block);
        }
        const uint32_t word = (ord & 3) == 0 ? w.x : ((ord & 3) == 1 ? w.y : ((ord & 3) == 2 ? w.z : w.w));
        // lower bound of the free flight: the same logf of the same argument the exact test uses, times a density
        // bound rounded toward zero, less two ulps for the products (u = 0: an infinite flight)
        const float flight_lb = inv_density_lb * (-logf(u01f(word))) * 0.999999f;
        if (flight_lb > seg_ub) continue;
        if (!have_slab) {
            make_slab(ray.o, ray.d, s);
            have_slab = true;
        }
        float tn;
        // the medium's segment is clipped to [tmin, best.t] (hittable.rs:754-761): its box bounds the segment
        if (!slab(s, lo.x, hi.x, lo.y, hi.y, lo.z, hi.z, __double2float_rd(tmin), __double2float_ru(best.t), tn)) continue;
        const int32_t ri = __float_as_int(lo.w);
        double t;
        if (medium_candidate<false>(sc, ri, ray, tmin, best.t, u01d(word), stack, t, tally)) {
            best.t = t;
            best.rec = ri;
            best.chain = 0;
        }
    }
}

// kPerlinShared (RTX_PERLIN_SMEM=1, scenes with exactly one Perlin table): the 4.75 KB table — 256 gradients and the three
// byte permutations (noise.rs:5-29) — is staged in shared memory by every CTA and NoiseTexture::value reads it there.
// kAdaptive (rtx_render_adaptive, adaptive.cuh): the dispenser's tiles are the entries of a.adaptive.tile_list, and a
// finished path with an odd sample index is also added to a.adaptive.aux.
// kEnv (a scene with an environment map): a miss adds env_lookup(a.env, d) instead of the constant background.
template <bool kCount, bool kPerlinShared = false, bool kOrder = false, bool kAdaptive = false>
__global__ void __launch_bounds__(kShadeBlock, WF_SHADE_MINB*(128 / kShadeBlock)) wf_shade2_kernel(WfArgs a, float4* __restrict__ accum, unsigned int* active_out,
                                                                                                   Counters* counters) {
    constexpr bool kEnv = false;
#include "shade2_body.cuh"
}

// The shade kernel of a scene with an environment map: not counted and without ray ordering (rtx_render_counted and
// RTX_ORDER=1 refuse such scenes). kCount and kOrder are template parameters only so that the body's `if constexpr`
// branches on them are discarded rather than compiled.
template <bool kPerlinShared, bool kAdaptive, bool kCount = false, bool kOrder = false>
__global__ void __launch_bounds__(kShadeBlock, WF_SHADE_MINB*(128 / kShadeBlock)) wf_shade2_env_kernel(WfArgs a, float4* __restrict__ accum, unsigned int* active_out,
                                                                                                       Counters* counters) {
    static_assert(!kCount && !kOrder, "no counted or ordered environment-map kernel");
    constexpr bool kEnv = true;
#include "shade2_body.cuh"
}

}  // namespace rtx
