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
template <bool kCount, bool kPerlinShared = false, bool kOrder = false, bool kAdaptive = false>
__global__ void __launch_bounds__(kShadeBlock, WF_SHADE_MINB*(128 / kShadeBlock)) wf_shade2_kernel(WfArgs a, float4* __restrict__ accum, unsigned int* active_out,
                                                                                                   Counters* counters) {
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int i = blockIdx.x * blockDim.x + tid;
    const bool valid = i < a.n_slots;
    int32_t stack[kStackSize];  // only a ConstantMedium with a general boundary traverses here
    Tally<kCount> tally;

    int bounce = valid ? a.pool.bounce[i] : -2;
    const bool dry = __ldcg(a.next_item) >= a.total_items;  // read now, needed after the shading: its latency is covered
    if constexpr (kPerlinShared) {
        __shared__ DPerlin s_perlin;
        static_assert(sizeof(DPerlin) % 16 == 0, "DPerlin is copied in 16-byte words");
        const uint4* src = reinterpret_cast<const uint4*>(a.sc.perlins);
        uint4* dst = reinterpret_cast<uint4*>(&s_perlin);
        for (int k = tid; k < (int)(sizeof(DPerlin) / 16); k += kShadeBlock) dst[k] = __ldg(src + k);
        __syncthreads();
        a.sc.perlins = &s_perlin;
    }

    // ---- shade: media first (a scatter point in front of the surface hit replaces it), then one level of color() ----
    RayD ray{mk(0, 0, 0), mk(0, 0, 1), 0.0};
    PathColor pc{1.f, 1.f, 1.f, 0.f, 0.f, 0.f};
    Sampler smp{a.k0, a.k1, 0u, 0u, 0u};
    bool fresh = false;
    int32_t src_rec = -1;  // the record the new ray starts on (kOrder)
    if (bounce >= 0) {
        ray.o = mk(a.pool.ox[i], a.pool.oy[i], a.pool.oz[i]);
        ray.d = mk(a.pool.dx[i], a.pool.dy[i], a.pool.dz[i]);
        ray.time = a.pool.time[i];
        Best best{a.pool.best_t[i], a.pool.best_rec[i], a.pool.best_chain[i]};
        pc = PathColor{a.pool.thr_r[i], a.pool.thr_g[i], a.pool.thr_b[i], 0.f, 0.f, 0.f};
        smp.pixel = a.pool.pixel[i];
        smp.sample = a.pool.sample[i];
        smp.bounce = (uint32_t)bounce;
        if (a.sc.n_media > 0) media_after(a.sc, ray, 0.001, best, smp, stack, tally);
        Albedo al;
        const bool ended = shade_hit<false, kPerlinShared>(a.sc, a.cam.background, a.max_depth, ray, best, smp, pc, bounce, al);
        apply_albedo(pc, al);
        if (ended) {
            atomicAdd(accum + smp.pixel, make_float4(pc.rad_r, pc.rad_g, pc.rad_b, 1.0f));  // one path sample done
            if constexpr (kAdaptive)
                if (smp.sample & 1u) atomicAdd(a.adaptive.aux + smp.pixel, make_float4(pc.rad_r, pc.rad_g, pc.rad_b, 1.0f));
            bounce = -1;
            a.pool.bounce[i] = -1;
        } else {
            fresh = true;
            src_rec = best.rec;
        }
    }
    {   // ---- refill empty slots per warp: consecutive items are the 32 pixels of one 8x4 tile at one sample index ----
        const bool want = bounce == -1;
        unsigned m = dry ? 0u : __ballot_sync(FULL, want);
        if (m != 0) {
            const int leader = __ffs(m) - 1;
            unsigned long long base = 0;
            if (lane == leader) base = atomicAdd(a.next_item, (unsigned long long)__popc(m));
            base = __shfl_sync(FULL, base, leader);
            const unsigned long long item = base + (unsigned long long)__popc(m & ((1u << lane) - 1u));
            if (want && item < a.total_items) {
                const unsigned long long group = item >> 5;
                const unsigned int tile = (unsigned int)(group / (unsigned long long)a.spp_count);
                const unsigned int smp_i = (unsigned int)(group - (unsigned long long)tile * (unsigned long long)a.spp_count);
                int tx, ty;
                tile_of_order(kAdaptive ? __ldg(a.adaptive.tile_list + tile) : tile, a.tiles_x, a.tiles_y, a.inv_per_block_row, tx, ty);
                const int pi = (int)(item & 31ull);
                const int px = tx * kTileW + (pi & (kTileW - 1));
                const int row = ty * kTileH + (pi / kTileW);  // row 0 = top
                if (px < a.width && row < a.height) {
                    smp.pixel = (uint32_t)(row * a.width + px);
                    smp.sample = (uint32_t)a.spp_begin + smp_i;
                    smp.bounce = 0;
                    camera_ray(a.cam, a.width, a.height, px, a.height - 1 - row, smp, ray);
                    pc = PathColor{1.f, 1.f, 1.f, 0.f, 0.f, 0.f};
                    bounce = 0;
                    fresh = true;
                }
            }
        }
    }
    // ---- the new ray goes to the pool with nothing hit yet: the trace kernel searches [0.001, inf) ----
    if (fresh) {
        a.pool.ox[i] = ray.o.x; a.pool.oy[i] = ray.o.y; a.pool.oz[i] = ray.o.z;
        a.pool.dx[i] = ray.d.x; a.pool.dy[i] = ray.d.y; a.pool.dz[i] = ray.d.z;
        a.pool.time[i] = ray.time;
        a.pool.best_t[i] = 1.7976931348623157e308; a.pool.best_rec[i] = -1; a.pool.best_chain[i] = 0;
        a.pool.thr_r[i] = pc.thr_r; a.pool.thr_g[i] = pc.thr_g; a.pool.thr_b[i] = pc.thr_b;
        a.pool.pixel[i] = smp.pixel; a.pool.sample[i] = smp.sample;
        a.pool.bounce[i] = bounce;
    }
    if constexpr (kOrder) {  // this slot's place in the next trace pass (order.cuh)
        uint2 kr = make_uint2(kOrderDead, 0u);
        if (fresh) kr.x = order_key(a.order, src_rec, ray.d.x, ray.d.y, ray.d.z);
        {   // one atomic per distinct key of the warp (camera rays of a refill share theirs: 32 same-address atomics
            // per warp cost the shade pass +50 us on every scene when each lane did its own)
            const unsigned same = __match_any_sync(FULL, kr.x);
            const int leader = __ffs(same) - 1;
            uint32_t base = 0;
            if (fresh && lane == leader) base = atomicAdd(a.order.hist + kr.x, (uint32_t)__popc(same));
            base = __shfl_sync(FULL, base, leader);
            kr.y = base + (uint32_t)__popc(same & ((1u << lane) - 1u));
        }
        if (valid) a.order.key_rank[i] = kr;
        order_scan_by_last_cta<kShadeBlock>(a.order, tid);
    }
    if (active_out) {
        const unsigned am = __ballot_sync(FULL, fresh);
        if (lane == 0 && am != 0) atomicAdd(active_out, (unsigned int)__popc(am));
    }
    if constexpr (kCount) {
        uint32_t v = tally.n_med;
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(FULL, v, off);
        if (lane == 0 && v) atomicAdd(&counters->medium_tests, (unsigned long long)v);
    }
}

}  // namespace rtx
