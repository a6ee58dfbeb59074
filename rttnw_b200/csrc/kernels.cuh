// kernels.cuh — device code of the rttnw hot path for sm_100a.
//
//   K1  trace_rays_kernel : every Hittable::hit + Bound::hit of src/math/hittable.rs / bound.rs
//   K2a wf_shade_kernel   : render()'s pixel loop + one level of color() + Material::scatter/emitted +
//                           Texture::value (src/main.rs:26-45,202-217, material.rs, texture.rs, noise.rs)
//   K2b wf_trace_kernel   : the closest surface hit of every ray in flight (the wavefront's other half)
//       render_kernel     : the same path loop as ONE kernel (megakernel; kept for the comparison in DESIGN.md)
//   K3  tonemap_kernel    : mean / sqrt / clamp / quantise (src/main.rs:217-225)
//       reduce_tonemap_peers_kernel : K3 fused with the multi-GPU sum over NVLink peer pointers
//
// The reference recurses through trait objects in f64. Here: an iterative while-while BVH
// traversal in world space (fp32 conservative slab tests on 64-byte nodes, exact-form f64
// primitive tests on 96-byte records; a primitive under Translate / YRotate wrappers pushes the
// ray through its composed transform chain first), hit records finalised once per query
// (including the Translate/YRotate post-processing of hittable.rs:606-613,699-712 exactly as
// written, Q13/Q14), an iterative path loop and Philox4x32-10 counters for every random draw.
#pragma once
#ifndef K1_MINB
#define K1_MINB 5  // 96 registers: 4.8 / 4.3 / 4.2 Grays/s on primary / secondary / tertiary rays of scene 9 (4, 6, 7 CTAs per SM: 4.3, 4.3, 4.5 on primaries)
#endif
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../include/rttnw_b200.h"
#include "device_types.h"
#include "order.cuh"

namespace rtx {

// ---------------------------------------------------------------------------
// small vector helpers
// ---------------------------------------------------------------------------
__device__ __forceinline__ double ldg_d(const double* p) { return __ldg(p); }

struct d3 {
    double x, y, z;
};
__device__ __forceinline__ d3 mk(double x, double y, double z) { return d3{x, y, z}; }
__device__ __forceinline__ d3 operator+(d3 a, d3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ d3 operator-(d3 a, d3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ d3 operator*(double s, d3 a) { return mk(s * a.x, s * a.y, s * a.z); }
__device__ __forceinline__ d3 operator-(d3 a) { return mk(-a.x, -a.y, -a.z); }
__device__ __forceinline__ double dot(d3 a, d3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ double comp(d3 a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }

struct RayD {
    d3 o, d;
    double time;
};

// ---------------------------------------------------------------------------
// Philox4x32-10 (counter based; replaces rand::thread_rng(), SURVEY §2.4).
// counter = (pixel, sample, bounce << 8 | purpose, block), key = seed.
// ---------------------------------------------------------------------------
enum Purpose : uint32_t { P_CAMERA = 0, P_LENS = 1, P_SCATTER = 2, P_MEDIUM = 3 };

__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0;
        uint32_t n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ float u01f(uint32_t w) { return (float)(w >> 8) * (1.0f / 16777216.0f); }
__device__ __forceinline__ double u01d(uint32_t w) { return (double)(w >> 8) * (1.0 / 16777216.0); }

struct Sampler {
    uint32_t k0, k1, pixel, sample, bounce;
    __device__ __forceinline__ uint4 block(Purpose p, uint32_t j) const {
        return philox4x32_10(pixel, sample, (bounce << 8) | (uint32_t)p, j, k0, k1);
    }
};

// ---------------------------------------------------------------------------
// Work counters (rtx_trace_rays_stats)
// ---------------------------------------------------------------------------
struct Counters {
    unsigned long long box_tests, node_visits, sphere_tests, rect_tests, instance_enters, medium_tests;
};
template <bool kCount>
struct Tally {
    __device__ __forceinline__ void node() {}
    __device__ __forceinline__ void sphere() {}
    __device__ __forceinline__ void rect() {}
    __device__ __forceinline__ void medium() {}
};
template <>
struct Tally<true> {
    uint32_t n_node = 0, n_sphere = 0, n_rect = 0, n_med = 0;
    __device__ __forceinline__ void node() { ++n_node; }
    __device__ __forceinline__ void sphere() { ++n_sphere; }
    __device__ __forceinline__ void rect() { ++n_rect; }
    __device__ __forceinline__ void medium() { ++n_med; }
};

// ---------------------------------------------------------------------------
// The fp32 half of a ray in the space currently being traversed: directed-rounding slab
// parameters for the BVH boxes (world space). The f64 half (origin, direction) is the ray itself,
// pushed through a primitive's transform chain when that primitive is tested (test_geometry).
// ---------------------------------------------------------------------------
struct SlabRay {
    float idx, idy, idz;     // fp32 1/d, magnitude clamped to 2^100
    float anx, any, anz;     // near offsets: round-down of -o * idx
    float afx, afy, afz;     // far offsets:  round-up   of -o * idx
};

__device__ __forceinline__ float clamp_inv(float d) {
    float inv = 1.0f / d;
    if (!(fabsf(inv) <= 0x1p100f)) inv = copysignf(0x1p100f, d);
    return inv;
}
__device__ __forceinline__ void make_slab(d3 o, d3 d, SlabRay& s) {
    s.idx = clamp_inv((float)d.x);
    s.idy = clamp_inv((float)d.y);
    s.idz = clamp_inv((float)d.z);
    double ax = -o.x * (double)s.idx, ay = -o.y * (double)s.idy, az = -o.z * (double)s.idz;
    s.anx = __double2float_rd(ax); s.afx = __double2float_ru(ax);
    s.any = __double2float_rd(ay); s.afy = __double2float_ru(ay);
    s.anz = __double2float_rd(az); s.afz = __double2float_ru(az);
}

// Conservative fp32 version of Bound::hit (bound.rs:13-32): never rejects a box the f64
// test would accept. lo/hi are rounded outward at build time, the offsets are rounded
// outward per ray, and the interval is widened by 2^-21 relative for the fma / reciprocal
// roundings. Returns the (widened) entry distance through `tnear`.
__device__ __forceinline__ bool slab(const SlabRay& s, float lox, float hix, float loy, float hiy, float loz, float hiz,
                                     float tmin, float tmax, float& tnear) {
    bool sx = s.idx < 0.0f, sy = s.idy < 0.0f, sz = s.idz < 0.0f;  // negative direction: the near plane is the box's hi
    float nx = fmaf(sx ? hix : lox, s.idx, s.anx), fx = fmaf(sx ? lox : hix, s.idx, s.afx);
    float ny = fmaf(sy ? hiy : loy, s.idy, s.any), fy = fmaf(sy ? loy : hiy, s.idy, s.afy);
    float nz = fmaf(sz ? hiz : loz, s.idz, s.anz), fz = fmaf(sz ? loz : hiz, s.idz, s.afz);
    float tn = fmaxf(fmaxf(nx, ny), nz);
    float tf = fminf(fminf(fx, fy), fz);
    tn = fmaf(-fabsf(tn), 0x1p-21f, tn);
    tf = fmaf(fabsf(tf), 0x1p-21f, tf);
    tnear = tn;
    return fmaxf(tn, tmin) <= fminf(tf, tmax);
}

__device__ __forceinline__ void apply_op(const XformOp& op, d3& o, d3& d) {
    if (op.kind == XF_TRANSLATE) {  // Translate::hit, hittable.rs:600-604
        o = mk(o.x - op.v[0], o.y - op.v[1], o.z - op.v[2]);
    } else {  // YRotate::hit, hittable.rs:687-692
        double sn = op.v[0], cs = op.v[1];
        o = mk(cs * o.x - sn * o.z, o.y, sn * o.x + cs * o.z);
        d = mk(cs * d.x - sn * d.z, d.y, sn * d.x + cs * d.z);
    }
}
// The ray in the object space of chain `chain` (an index into SceneView::chains; 0 = world): the
// composition of the wrappers' Translate::hit / YRotate::hit ray transforms, applied in one step.
__device__ __forceinline__ void to_space(const SceneView& sc, int32_t chain, d3& o, d3& d) {
    const double2* cp = reinterpret_cast<const double2*>(sc.chains + chain);
    double2 r = __ldg(cp), t0 = __ldg(cp + 1);
    double tz = ldg_d(&sc.chains[chain].tz);
    o = mk(r.x * o.x - r.y * o.z + t0.x, o.y + t0.y, r.y * o.x + r.x * o.z + tz);
    d = mk(r.x * d.x - r.y * d.z, d.y, r.y * d.x + r.x * d.z);
}

// ---------------------------------------------------------------------------
// Primitive tests in f64, following the reference's formulas. They only decide and return t; the hit record is built
// once, for the winner. Two deliberate departures, each one rounding away from the reference and far inside the 1e-5
// contract (largest t error over 9 x 10^7 fixed rays: 1e-7, profiles/r2_parity.json): the sphere roots are multiplied
// by 1 / a where hittable.rs:97,102 divides by a, and a MovingSphere's centre uses a stored 1 / (t1 - t0). A root that
// lands within that rounding of t_min / t_max can therefore be accepted on one side and rejected on the other: such
// rays are what the oracle's grazing-tie flag marks, and ids are compared outside that set.
// ---------------------------------------------------------------------------
// Sphere::hit / MovingSphere::hit quadratic, hittable.rs:88-108,196-216 (Q9: both ends inclusive)
__device__ __forceinline__ bool sphere_roots(d3 o, d3 d, d3 c, double r, double tmin, double tmax, double& t) {
    d3 oc = o - c;
    double a = dot(d, d);
    double half_b = dot(oc, d);
    double cc = dot(oc, oc) - r * r;
    double disc = half_b * half_b - a * cc;
    if (disc < 0.0) return false;
    double sq = sqrt(disc);
    double inv_a = 1.0 / a;
    double root = (-half_b - sq) * inv_a;
    if (root < tmin || tmax < root) {
        root = (-half_b + sq) * inv_a;
        if (root < tmin || tmax < root) return false;
    }
    t = root;
    return true;
}
__device__ __forceinline__ d3 msphere_center(const double* d, double time) {  // hittable.rs:187-191
    double f = (time - d[7]) * d[8];
    return mk(d[0] + f * d[3], d[1] + f * d[4], d[2] + f * d[5]);
}
// Rectangle::hit, hittable.rs:503-513 (Q11: t inclusive, ranges half-open, NaN never contained)
__device__ __forceinline__ bool rect_hit(d3 o, d3 d, int plane, const double* r, double tmin, double tmax, double& t) {
    int a0 = plane == 2 ? 1 : 0, a1 = plane == 0 ? 1 : 2, ak = plane == 0 ? 2 : (plane == 1 ? 1 : 0);
    double tt = (r[4] - comp(o, ak)) / comp(d, ak);
    if (tt < tmin || tt > tmax) return false;
    double p0 = comp(o, a0) + tt * comp(d, a0);
    double p1 = comp(o, a1) + tt * comp(d, a1);
    if (!(r[0] <= p0 && p0 < r[1]) || !(r[2] <= p1 && p1 < r[3])) return false;
    t = tt;
    return true;
}

struct Best {
    double t;       // closest accepted distance so far (the `closest` of List::hit, hittable.rs:155)
    int32_t rec;    // record index, -1 = none
    int32_t chain;  // transform chain of the record that was hit (index into SceneView::chains; 0 = none)
};

constexpr int kStackSize = kTraversalStack;
constexpr int32_t kSentinel = (int32_t)0x80000000;       // bottom of a query's stack

// One geometric record (sphere / moving sphere / rectangle / box) against the ray: the ray is pushed
// through the record's wrapper chain first (Translate::hit / YRotate::hit, hittable.rs:600-604,687-692).
// `hit_rec` is the record the hit record is built from (a box reports the rectangle of the face hit).
// One copy of each intersection routine per kernel: code size is what the instruction cache sees.
template <bool kCount>
__device__ __forceinline__ bool test_geometry(const SceneView& sc, int32_t ri, int4 h, const RayD& ray, double tmin, double tmax,
                                              double& t, int32_t& hit_rec, Tally<kCount>& tally) {
    const double* q = sc.records[ri].d;
    d3 o = ray.o, d = ray.d;
    if (h.w != 0) to_space(sc, h.w, o, d);
    double2 a = __ldg(reinterpret_cast<const double2*>(q)), b = __ldg(reinterpret_cast<const double2*>(q + 2));
    hit_rec = ri;
    if (h.x <= REC_MSPHERE) {
        tally.sphere();
        d3 c = mk(a.x, a.y, b.x);
        double r = b.y;
        if (h.x == REC_MSPHERE) {  // MovingSphere::center, hittable.rs:187-191
            double2 e = __ldg(reinterpret_cast<const double2*>(q + 4)), g = __ldg(reinterpret_cast<const double2*>(q + 6));
            double f = (ray.time - g.y) * ldg_d(q + 8);
            c = mk(a.x + f * b.y, a.y + f * e.x, b.x + f * e.y);
            r = g.x;
        }
        return sphere_roots(o, d, c, r, tmin, tmax, t);
    }
    tally.rect();
    if (h.x == REC_BOX) {
        // Cube::hit = List::hit over six rectangles (hittable.rs:580-582): a line meets them where it enters and
        // where it leaves the box, at the (k - o) / d each Rectangle::hit computes (:504); the closest one inside
        // [tmin, tmax] is the entry face, or the exit face when the entry lies before tmin.
        double2 e = __ldg(reinterpret_cast<const double2*>(q + 4));
        const double lo[3] = {a.x, a.y, b.x}, hi[3] = {b.y, e.x, e.y};
        double tn = -CUDART_INF, tf = CUDART_INF;
        int fn = 0, ff = 0;
#pragma unroll
        for (int ax = 0; ax < 3; ++ax) {
            const double oa = comp(o, ax), da = comp(d, ax);
            const double t0 = (lo[ax] - oa) / da, t1 = (hi[ax] - oa) / da;
            const bool neg = t1 < t0;  // the ray runs from hi to lo on this axis
            const double tnear = neg ? t1 : t0, tfar = neg ? t0 : t1;
            const int base = ax == 0 ? 4 : (ax == 1 ? 2 : 0);  // Cube::new order: xy(min.z), xy(max.z), xz(min.y), xz(max.y), yz(min.x), yz(max.x)
            if (tnear > tn) { tn = tnear; fn = base + (neg ? 1 : 0); }
            if (tfar < tf) { tf = tfar; ff = base + (neg ? 0 : 1); }
        }
        if (!(tn <= tf)) return false;
        double tt = tn;
        int face = fn;
        if (tn < tmin) { tt = tf; face = ff; }
        if (tt < tmin || tt > tmax) return false;
        t = tt;
        hit_rec = h.y + face;
        return true;
    }
    double dd[5] = {a.x, a.y, b.x, b.y, ldg_d(q + 4)};
    return rect_hit(o, d, h.x - REC_RECT_XY, dd, tmin, tmax, t);
}

// One inner node: both child boxes against the ray; returns the next node to visit and pushes the
// farther child when both are hit.
// (Asking the deferred child into the L2 when it is pushed — prefetch.global.L2, the one fetch of the loop whose address
// is known early — was measured on the 2*10^6-sphere scene, 368 MB against 126 MB of L2: 9.13 ms against 9.02 ms for
// 2*10^6 rays, and -3 % on scene 9. Not kept.)
template <bool kCount>
__device__ __forceinline__ int32_t node_step(const SceneView& sc, int32_t cur, const SlabRay& s, float tmin_f, float tmax_f,
                                             int32_t* stack, int& sp, Tally<kCount>& tally) {
    const float4* np = reinterpret_cast<const float4*>(sc.nodes + cur);
    float4 q0 = __ldg(np), q1 = __ldg(np + 1), q2 = __ldg(np + 2);
    int4 meta = __ldg(reinterpret_cast<const int4*>(np + 3));
    tally.node();
    float n0, n1;
    bool h0 = slab(s, q0.x, q0.y, q0.z, q0.w, q2.x, q2.y, tmin_f, tmax_f, n0);
    bool h1 = slab(s, q1.x, q1.y, q1.z, q1.w, q2.z, q2.w, tmin_f, tmax_f, n1);
    if (h0 && h1) {
        bool swap = n1 < n0;
        stack[sp++] = swap ? meta.x : meta.y;
        return swap ? meta.y : meta.x;
    }
    if (h0) return meta.x;
    if (h1) return meta.y;
    return stack[--sp];
}

// Closest hit over the BVH rooted at `root` for `ray` in [tmin, best.t]: plain while-while
// traversal in world space. Used by the fixed-ray kernel, the wavefront trace kernel and
// ConstantMedium boundary queries. `stack` is a per-thread array, `sp` the first free slot.
template <bool kCount>
__device__ __forceinline__ void traverse_simple(const SceneView& sc, int32_t root, const RayD& ray, double tmin, Best& best,
                                                int32_t* stack, int sp, Tally<kCount>& tally) {
    SlabRay s;
    make_slab(ray.o, ray.d, s);
    float tmin_f = __double2float_rd(tmin);
    float tmax_f = __double2float_ru(best.t);
    stack[sp++] = kSentinel;
    int32_t cur = root;
    while (true) {
        while (cur >= 0) cur = node_step(sc, cur, s, tmin_f, tmax_f, stack, sp, tally);
        if (cur == kSentinel) break;
        int32_t v = ~cur;
        int32_t first = v >> 4, count = v & 15;
        cur = stack[--sp];
        for (int32_t i = 0; i < count; ++i) {
            int4 h = __ldg(reinterpret_cast<const int4*>(sc.records + first + i));
            double t;
            int32_t hit_rec;
            if (test_geometry(sc, first + i, h, ray, tmin, best.t, t, hit_rec, tally)) {
                best.t = t;
                best.rec = hit_rec;
                best.chain = h.w;
                tmax_f = __double2float_ru(t);
            }
        }
    }
}

// Opt-in (RTX_BVH_WIDE=1): the same query over the 4-wide copy of the world BVH (flatten.cpp emit_wide). A node is
// two consecutive 64-byte entries: four child boxes are tested per step, the hits ordered by entry distance with a
// five-exchange network, the nearest entered and the others deferred farthest first. Half the dependent fetches of
// the binary loop per leaf reached, but 140 SASS instructions per step against 68, and all four boxes are tested
// where the binary loop prunes a pair with its parent: measured 536 M samples/s against 600 M on scene 9 (same
// hits: tests/test_gpu_parity.py::test_wide_bvh_traversal_finds_the_same_hits). Not the default.
__device__ __forceinline__ void order2(float& ta, int32_t& ra, float& tb, int32_t& rb) {
    const bool sw = tb < ta;
    const float t = sw ? tb : ta;
    const int32_t r = sw ? rb : ra;
    tb = sw ? ta : tb;
    rb = sw ? ra : rb;
    ta = t;
    ra = r;
}
template <bool kCount>
__device__ __forceinline__ void traverse_wide(const SceneView& sc, int32_t root, const RayD& ray, double tmin, Best& best,
                                              int32_t* stack, Tally<kCount>& tally) {
    SlabRay s;
    make_slab(ray.o, ray.d, s);
    const float tmin_f = __double2float_rd(tmin);
    float tmax_f = __double2float_ru(best.t);
    int32_t* top = stack;
    *top++ = kSentinel;
    int32_t cur = root;
    const float kMiss = __int_as_float(0x7f800000);  // +inf
    while (true) {
        while (cur >= 0) {
            const float4* np = reinterpret_cast<const float4*>(sc.nodes + cur);
            float t0, t1, t2, t3;
            int32_t r0, r1, r2, r3;
            {
                float4 q0 = __ldg(np), q1 = __ldg(np + 1), q2 = __ldg(np + 2);
                int4 meta = __ldg(reinterpret_cast<const int4*>(np + 3));
                bool h0 = slab(s, q0.x, q0.y, q0.z, q0.w, q2.x, q2.y, tmin_f, tmax_f, t0);
                bool h1 = slab(s, q1.x, q1.y, q1.z, q1.w, q2.z, q2.w, tmin_f, tmax_f, t1);
                t0 = h0 ? t0 : kMiss; t1 = h1 ? t1 : kMiss;
                r0 = meta.x; r1 = meta.y;
            }
            {
                float4 q0 = __ldg(np + 4), q1 = __ldg(np + 5), q2 = __ldg(np + 6);
                int4 meta = __ldg(reinterpret_cast<const int4*>(np + 7));
                bool h2 = slab(s, q0.x, q0.y, q0.z, q0.w, q2.x, q2.y, tmin_f, tmax_f, t2);
                bool h3 = slab(s, q1.x, q1.y, q1.z, q1.w, q2.z, q2.w, tmin_f, tmax_f, t3);
                t2 = h2 ? t2 : kMiss; t3 = h3 ? t3 : kMiss;
                r2 = meta.x; r3 = meta.y;
            }
            tally.node();
            tally.node();  // two 64-byte entries, four box tests
            order2(t0, r0, t1, r1);
            order2(t2, r2, t3, r3);
            order2(t0, r0, t2, r2);
            order2(t1, r1, t3, r3);
            order2(t1, r1, t2, r2);
            // ascending now, the misses (+inf) last: defer the far hits, farthest first
            if (t3 < kMiss) *top++ = r3;
            if (t2 < kMiss) *top++ = r2;
            if (t1 < kMiss) *top++ = r1;
            cur = t0 < kMiss ? r0 : *--top;
        }
        if (cur == kSentinel) break;
        int32_t v = ~cur;
        int32_t first = v >> 4, count = v & 15;
        cur = *--top;
        for (int32_t i = 0; i < count; ++i) {
            int4 h = __ldg(reinterpret_cast<const int4*>(sc.records + first + i));
            double t;
            int32_t hit_rec;
            if (test_geometry(sc, first + i, h, ray, tmin, best.t, t, hit_rec, tally)) {
                best.t = t;
                best.rec = hit_rec;
                best.chain = h.w;
                tmax_f = __double2float_ru(t);
            }
        }
    }
}

// ConstantMedium::hit, hittable.rs:740-796 (Q16), for the medium record `ri`: the scatter distance as
// a candidate in [tmin, tmax]. `u` is the uniform variate the reference draws at :765.
template <bool kPrecise, bool kCount>
__device__ __forceinline__ bool medium_candidate(const SceneView& sc, int32_t ri, const RayD& ray, double tmin, double tmax, double u,
                                                 int32_t* stack, double& t, Tally<kCount>& tally) {
    const Record* rp = sc.records + ri;
    int4 h = __ldg(reinterpret_cast<const int4*>(rp));
    const double* q = rp->d;
    tally.medium();
    double r1, r2;
    if (h.w == -1) {
        // boundary = one untransformed sphere: hit(-inf, inf) is the near root, hit(t1 + 1e-4, inf) the far
        // root if it clears t1 + 1e-4 (Sphere::hit tries the near root first; it is below the new t_min)
        d3 c = mk(ldg_d(q + 4), ldg_d(q + 5), ldg_d(q + 6));
        double rad = ldg_d(q + 7);
        d3 oc = ray.o - c;
        double a = dot(ray.d, ray.d), half_b = dot(oc, ray.d), cc = dot(oc, oc) - rad * rad;
        double disc = half_b * half_b - a * cc;
        if (disc < 0.0) return false;
        double sq = sqrt(disc);
        double inv_a = 1.0 / a;
        r1 = (-half_b - sq) * inv_a;
        r2 = (-half_b + sq) * inv_a;
        if (r2 < r1 + 0.0001) return false;
    } else if (h.w <= -2) {
        // boundary = one Cube under a wrapper chain: the line meets its six rectangles where it enters and
        // where it leaves the box, at the same (k - o) / d each Rectangle::hit computes (hittable.rs:504)
        d3 o = ray.o, dd = ray.d;
        if (h.w != -2) to_space(sc, -2 - h.w, o, dd);
        r1 = -CUDART_INF;
        r2 = CUDART_INF;
#pragma unroll
        for (int ax = 0; ax < 3; ++ax) {
            double oa = comp(o, ax), da = comp(dd, ax);
            double t0 = (ldg_d(q + 4 + ax) - oa) / da, t1 = (ldg_d(q + 7 + ax) - oa) / da;
            r1 = fmax(r1, fmin(t0, t1));
            r2 = fmin(r2, fmax(t0, t1));
        }
        if (!(r1 < r2) || r2 < r1 + 0.0001) return false;
    } else {
        // boundary.hit(ray, -inf, inf) then boundary.hit(ray, t1 + 1e-4, inf), hittable.rs:745-752
        r1 = r2 = 0.0;
        double from = -CUDART_INF;
#pragma unroll 1
        for (int pass = 0; pass < 2; ++pass) {
            Best b{CUDART_INF, -1, 0};
            traverse_simple(sc, h.w, ray, from, b, stack, 0, tally);
            if (b.rec < 0) return false;
            if (pass == 0) { r1 = b.t; from = r1 + 0.0001; } else { r2 = b.t; }
        }
    }
    r1 = fmax(r1, tmin);
    r2 = fmin(r2, tmax);
    if (!(r1 < r2)) return false;
    r1 = fmax(r1, 0.0);
    double len = sqrt(dot(ray.d, ray.d));
    double inside = (r2 - r1) * len;
    double hit_distance = kPrecise ? ldg_d(q) * log(u) : ldg_d(q) * (double)logf((float)u);
    if (hit_distance > inside) return false;
    t = r1 + hit_distance / len;
    return true;
}

// Every medium the ray can reach, before the surface traversal: the scatter point is a candidate
// like any surface hit and the closest candidate wins — the same answer the reference's
// `closest`-clipped ConstantMedium::hit gives in whatever order List::hit meets it. `smp` != null:
// medium number k draws word (k & 3) of Philox block (MEDIUM, k >> 2); else `xi` is the variate.
template <bool kPrecise, bool kCount>
__device__ __forceinline__ void media_prepass(const SceneView& sc, const RayD& ray, const SlabRay& s, double tmin, Best& best,
                                              double xi, const Sampler* smp, int32_t* stack, Tally<kCount>& tally) {
    float tmin_f = __double2float_rd(tmin);
    uint4 w = make_uint4(0, 0, 0, 0);
    int32_t w_block = -1;
    for (int32_t m = 0; m < sc.n_media; ++m) {
        const float4* mp = reinterpret_cast<const float4*>(sc.media + m);
        float4 lo = __ldg(mp), hi = __ldg(mp + 1);
        float tn;
        // the medium's segment is clipped to [tmin, best.t] (hittable.rs:754-761): its box bounds the segment
        if (!slab(s, lo.x, hi.x, lo.y, hi.y, lo.z, hi.z, tmin_f, __double2float_ru(best.t), tn)) continue;
        int32_t ri = __float_as_int(lo.w);
        double u = xi;
        if (smp) {
            int32_t ord = (int32_t)ldg_d(sc.records[ri].d + 1);
            if ((ord >> 2) != w_block) {
                w_block = ord >> 2;
                w = smp->block(P_MEDIUM, (uint32_t)w_block);
            }
            uint32_t word = (ord & 3) == 0 ? w.x : ((ord & 3) == 1 ? w.y : ((ord & 3) == 2 ? w.z : w.w));
            u = u01d(word);
        }
        double t;
        if (medium_candidate<kPrecise>(sc, ri, ray, tmin, best.t, u, stack, t, tally)) {
            best.t = t;
            best.rec = ri;
            best.chain = 0;
        }
    }
}

// ---------------------------------------------------------------------------
// Hit record of the winning record (HitRecord, hittable.rs:15-27), built once.
// ---------------------------------------------------------------------------
struct HitOut {
    d3 p, n;       // point and (face-flipped, possibly Q14-mangled) normal
    d3 on;         // outward unit normal in object space (spheres: the argument of Sphere::uv)
    double u, v;   // when kPrecise; the render path computes them only for textures that look at them
    double ru, rv; // rectangles, render path: the in-plane coordinates (p0, p1) of the hit, for rect_uv()
    int32_t material;  // material index, or -(1 + texture) for a medium's Isotropic
    int32_t prim_id;
    int32_t type;
    bool front_face;
};

// Rectangle u, v (hittable.rs:515-516) from the in-plane hit coordinates finalize_hit<false> left in ru, rv
__device__ __forceinline__ void rect_uv(const SceneView& sc, int32_t rec, double p0, double p1, float& u, float& v) {
    const double* d = sc.records[rec].d;
    double r0 = ldg_d(d), r1 = ldg_d(d + 1), r2 = ldg_d(d + 2), r3 = ldg_d(d + 3);
    u = (float)((p0 - r0) / (r1 - r0));
    v = (float)((p1 - r2) / (r3 - r2));
}

__device__ __forceinline__ void sphere_uv(d3 p, double& u, double& v) {  // hittable.rs:77-83
    const double PI = 3.14159265358979323846;
    double theta = acos(-p.y);
    double phi = atan2(-p.z, p.x) + PI;
    u = phi / (2.0 * PI);
    v = theta / PI;
}

template <bool kPrecise>
__device__ __forceinline__ void finalize_hit(const SceneView& sc, const RayD& ray, const Best& best, HitOut& out) {
    const Record* rp = sc.records + best.rec;
    int4 h = __ldg(reinterpret_cast<const int4*>(rp));
    const double* d = rp->d;
    int32_t chain = best.chain;
    if (h.x == REC_MEDIUM) chain = (int32_t)ldg_d(d + 2);
    d3 o = ray.o, dir = ray.d;
    int32_t begin = 0, len = 0;
    if (chain != 0) {
        to_space(sc, chain, o, dir);
        begin = sc.chains[chain].begin;
        len = sc.chains[chain].len;
    }
    double t = best.t;
    d3 p = o + t * dir;  // Ray::point_at_parameter in the primitive's own space
    d3 n;
    bool ff;
    out.u = 0.0;
    out.v = 0.0;
    out.ru = 0.0;
    out.rv = 0.0;
    out.type = h.x;
    out.prim_id = h.z;
    out.material = h.y;
    if (h.x == REC_MEDIUM) {  // hittable.rs:778-789: arbitrary normal, front_face = true, u = v = 0
        n = mk(1.0, 0.0, 0.0);
        ff = true;
        out.on = n;
        out.material = -(1 + h.y);
    } else {
        d3 outward;
        if (h.x <= REC_MSPHERE) {
            d3 c = mk(ldg_d(d), ldg_d(d + 1), ldg_d(d + 2));
            double r = ldg_d(d + 3);
            if (h.x == REC_MSPHERE) {  // MovingSphere::center, hittable.rs:187-191; u = v = 0 (Q10)
                double f = (ray.time - ldg_d(d + 7)) * ldg_d(d + 8);
                c = mk(c.x + f * r, c.y + f * ldg_d(d + 4), c.z + f * ldg_d(d + 5));
                r = ldg_d(d + 6);
            }
            if (kPrecise) {
                outward = mk((p.x - c.x) / r, (p.y - c.y) / r, (p.z - c.z) / r);  // hittable.rs:111,219
            } else {  // render path: one reciprocal (differs from the three divisions by one rounding)
                double ir = 1.0 / r;
                outward = mk((p.x - c.x) * ir, (p.y - c.y) * ir, (p.z - c.z) * ir);
            }
            if (kPrecise && h.x == REC_SPHERE) sphere_uv(outward, out.u, out.v);
        } else {
            int plane = h.x - REC_RECT_XY;
            int a0 = plane == 2 ? 1 : 0, a1 = plane == 0 ? 1 : 2;
            double r0 = ldg_d(d), r1 = ldg_d(d + 1), r2 = ldg_d(d + 2), r3 = ldg_d(d + 3);
            double p0 = comp(o, a0) + t * comp(dir, a0), p1 = comp(o, a1) + t * comp(dir, a1);
            if (kPrecise) {
                out.u = (p0 - r0) / (r1 - r0);  // hittable.rs:515-516
                out.v = (p1 - r2) / (r3 - r2);
            } else {  // two f64 divisions only an ImageTexture would look at: left to rect_uv()
                out.ru = p0;
                out.rv = p1;
            }
            outward = mk(plane == 2 ? 1.0 : 0.0, plane == 1 ? 1.0 : 0.0, plane == 0 ? 1.0 : 0.0);  // +k axis (Q11)
        }
        out.on = outward;
        ff = dot(dir, outward) < 0.0;  // HitRecord::face_normal, hittable.rs:30-44
        n = ff ? outward : -outward;
    }
    // unwind the wrappers, innermost first (what Translate::hit / YRotate::hit do on the way out)
    for (int32_t k = len - 1; k >= 0; --k) {
        XformOp op = sc.xforms[begin + k];
        if (op.kind == XF_ROTATE_Y) {
            double sn = op.v[0], cs = op.v[1];
            // Q14 (hittable.rs:700-705): [0] is overwritten first and the NEW [0] feeds [2]
            p.x = cs * p.x + sn * p.z;
            p.z = -sn * p.x + cs * p.z;
            n.x = cs * n.x + sn * n.z;
            n.z = -sn * n.x + cs * n.z;
            ff = dot(dir, n) < 0.0;  // against the object-space ray (hittable.rs:706)
            n = ff ? n : -n;
            dir = mk(cs * dir.x + sn * dir.z, dir.y, -sn * dir.x + cs * dir.z);  // direction one level out
        } else {
            ff = dot(dir, n) < 0.0;  // Q13 (hittable.rs:607): face_normal re-run on the flipped normal
            n = ff ? n : -n;
            p = mk(p.x + op.v[0], p.y + op.v[1], p.z + op.v[2]);
        }
    }
    out.p = p;
    out.n = n;
    out.front_face = ff;
}

// ---------------------------------------------------------------------------
// K1: fixed rays
// ---------------------------------------------------------------------------
template <bool kCount>
__global__ void __launch_bounds__(128, K1_MINB) trace_rays_kernel(SceneView sc, int64_t n, const rtx_ray* __restrict__ rays,
                                                         rtx_hit* __restrict__ hits, Counters* counters) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    Tally<kCount> tally;
    int32_t stack[kStackSize];
    if (i < n) {
        const double2* rp = reinterpret_cast<const double2*>(rays + i);  // 80 bytes = 5 x 16
        double2 a = __ldg(rp), b = __ldg(rp + 1), c = __ldg(rp + 2), d = __ldg(rp + 3), e = __ldg(rp + 4);
        RayD ray{mk(a.x, a.y, b.x), mk(b.y, c.x, c.y), d.x};
        double tmin = d.y, tmax = e.x, xi = e.y;
        Best best{tmax, -1, 0};
        SlabRay sr;
        make_slab(ray.o, ray.d, sr);
        media_prepass<true>(sc, ray, sr, tmin, best, xi, nullptr, stack, tally);
        traverse_simple(sc, sc.world_root, ray, tmin, best, stack, 0, tally);
        if (!kCount) {
            rtx_hit h;
            if (best.rec >= 0) {
                HitOut ho;
                finalize_hit<true>(sc, ray, best, ho);
                h.prim_id = ho.prim_id; h.material = ho.material; h.front_face = ho.front_face ? 1 : 0; h._pad = 0;
                h.t = best.t;
                h.p[0] = ho.p.x; h.p[1] = ho.p.y; h.p[2] = ho.p.z;
                h.normal[0] = ho.n.x; h.normal[1] = ho.n.y; h.normal[2] = ho.n.z;
                h.u = ho.u; h.v = ho.v;
            } else {
                h.prim_id = RTX_MISS; h.material = -1; h.front_face = 0; h._pad = 0;
                h.t = 0; h.p[0] = h.p[1] = h.p[2] = 0; h.normal[0] = h.normal[1] = h.normal[2] = 0; h.u = h.v = 0;
            }
            hits[i] = h;
        }
    }
    if constexpr (kCount) {
        // warp-reduce, one atomic per warp per counter
        uint32_t vals[4] = {tally.n_node, tally.n_sphere, tally.n_rect, tally.n_med};
#pragma unroll
        for (int k = 0; k < 4; ++k)
            for (int off = 16; off > 0; off >>= 1) vals[k] += __shfl_xor_sync(0xffffffffu, vals[k], off);
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&counters->node_visits, (unsigned long long)vals[0]);
            atomicAdd(&counters->box_tests, 2ull * vals[0]);
            atomicAdd(&counters->sphere_tests, (unsigned long long)vals[1]);
            atomicAdd(&counters->rect_tests, (unsigned long long)vals[2]);
            atomicAdd(&counters->medium_tests, (unsigned long long)vals[3]);
        }
    }
}

// ---------------------------------------------------------------------------
// Textures (src/math/texture.rs, noise.rs), fp32
// ---------------------------------------------------------------------------
struct f3 {
    float x, y, z;
};
__device__ __forceinline__ f3 mkf(float x, float y, float z) { return f3{x, y, z}; }

// kShared: `tab` is a copy staged in shared memory (plain loads), else the table in global memory (read-only path)
template <bool kShared = false>
__device__ __forceinline__ float perlin_noise(const DPerlin* __restrict__ tab, float px, float py, float pz) {  // noise.rs:49-94
    float fx = floorf(px), fy = floorf(py), fz = floorf(pz);
    float u = px - fx, v = py - fy, w = pz - fz;
    int i = (int)fx, j = (int)fy, k = (int)fz;
    float uu = u * u * (3.f - 2.f * u), vv = v * v * (3.f - 2.f * v), ww = w * w * (3.f - 2.f * w);
    float acc = 0.f;
#pragma unroll
    for (int di = 0; di < 2; ++di) {
        uint32_t hx = tab->perm[0][(i + di) & 255];
#pragma unroll
        for (int dj = 0; dj < 2; ++dj) {
            uint32_t hy = tab->perm[1][(j + dj) & 255];
#pragma unroll
            for (int dk = 0; dk < 2; ++dk) {
                uint32_t hz = tab->perm[2][(k + dk) & 255];
                const float4* gp = reinterpret_cast<const float4*>(tab->ranvec[hx ^ hy ^ hz]);
                float4 g = kShared ? *gp : __ldg(gp);
                float wu = di ? uu : 1.f - uu, wv = dj ? vv : 1.f - vv, wwt = dk ? ww : 1.f - ww;
                acc += wu * wv * wwt * (g.x * (u - di) + g.y * (v - dj) + g.z * (w - dk));
            }
        }
    }
    return acc;
}
template <bool kShared = false>
__device__ __forceinline__ float perlin_turbulence(const DPerlin* tab, float px, float py, float pz) {  // noise.rs:96-108, depth 7
    float acc = 0.f, weight = 1.f;
#pragma unroll 1
    for (int i = 0; i < 7; ++i) {
        acc += weight * perlin_noise<kShared>(tab, px, py, pz);
        weight *= 0.5f;
        px *= 2.f; py *= 2.f; pz *= 2.f;
    }
    return acc;
}

// CheckerTexture (texture.rs:15-30, Q21) selects a child; children may nest. Returns the texture that
// finally gets evaluated.
__device__ __forceinline__ DTexture resolve_texture(const SceneView& sc, int32_t ti, d3 p) {
    DTexture t = sc.textures[ti];
#pragma unroll 1
    for (int guard = 0; guard < 8 && t.kind == RTX_TEX_CHECKER; ++guard) {
        // f64 products keep the stripe edges of the radius-1000 ground sphere where the reference puts them;
        // one sinf call site (its large-argument reduction is ~500 instructions of code)
        float sines = 1.f;
#pragma unroll 1
        for (int c = 0; c < 3; ++c) sines *= sinf((float)(10.0 * comp(p, c)));
        t = sc.textures[sines < 0.f ? t.a : t.b];
    }
    return t;
}
// NoiseTexture::value, texture.rs:52-59 (Q22): grey 0.5 (1 + sin(scale z + 10 turb(p)))
template <bool kShared = false>
__device__ __forceinline__ float noise_value(const SceneView& sc, int32_t perlin, float scale, float px, float py, float pz) {
    float turb = perlin_turbulence<kShared>(sc.perlins + perlin, px, py, pz);
    return 0.5f * (1.f + sinf(scale * pz + 10.f * turb));
}
// Texture::value of a resolved texture. (u, v) are only meaningful when the texture's uses-uv flag is set.
template <bool kShared = false>
__device__ __forceinline__ f3 texture_eval(const SceneView& sc, const DTexture& t, float u, float v, d3 p) {
    if (t.kind == RTX_TEX_SOLID) return mkf(t.f[0], t.f[1], t.f[2]);
    if (t.kind == RTX_TEX_NOISE) {
        float g = noise_value<kShared>(sc, t.a, t.f[0], (float)p.x, (float)p.y, (float)p.z);
        return mkf(g, g, g);
    }
    if (t.kind == RTX_TEX_IMAGE) {  // texture.rs:77-106 (Q23): nearest texel, bytes / 255
        DImage img = sc.images[t.a];
        if (img.tex == 0) return mkf(0.f, 1.f, 1.f);
        float uu = fminf(fmaxf(u, 0.f), 1.f), vv = 1.f - fminf(fmaxf(v, 0.f), 1.f);
        int i = (int)(uu * (float)img.width), j = (int)(vv * (float)img.height);
        i = min(i, img.width - 1);
        j = min(j, img.height - 1);
        uchar4 px = tex2D<uchar4>((cudaTextureObject_t)img.tex, (float)i + 0.5f, (float)j + 0.5f);
        const float s = 1.0f / 255.0f;
        return mkf(px.x * s, px.y * s, px.z * s);
    }
    return mkf(0.f, 0.f, 0.f);
}

// Vec3f::random_in_unit_space, vec3.rs:149-160: candidate j = Philox block (SCATTER, j) words 0..2.
// The candidates are exact in fp32 and their squared length is exact in f64, so the accept /
// reject decisions are identical to the oracle's. `w3_first` returns word 3 of block 0
// (the Dielectric's uniform, material.rs:189).
__device__ __forceinline__ d3 random_in_unit_space(const Sampler& smp) {
    for (uint32_t j = 0;; ++j) {
        uint4 w = smp.block(P_SCATTER, j);
        double x = 2.0 * u01d(w.x) - 1.0, y = 2.0 * u01d(w.y) - 1.0, z = 2.0 * u01d(w.z) - 1.0;
        if (x * x + y * y + z * z < 1.0) return mk(x, y, z);
    }
}

// ---------------------------------------------------------------------------
// One level of color() (main.rs:26-45, Q7) for a ray whose closest hit is known: adds the emitted /
// background radiance, scatters (Material::scatter) and leaves the next ray in `ray`. Returns true
// when the path ends here. Shared by the megakernel's shade phase and the wavefront shade kernel.
// ---------------------------------------------------------------------------
struct PathColor {
    float thr_r, thr_g, thr_b;  // product of the attenuations so far
    float rad_r, rad_g, rad_b;  // radiance gathered so far
};

// What shade_hit leaves for the caller to apply: the texture value multiplies the throughput (scatter) or
// is added as emitted radiance. With kDeferNoise a Perlin texture is NOT evaluated here: `noise_perlin`
// >= 0 names the table and the caller evaluates noise_value(noise_perlin, noise_scale, p) — densely, for all
// the threads of the CTA that need it, instead of 7 octaves x 8 lattice corners on a mostly idle warp.
struct Albedo {
    float r, g, b;
    bool emissive;
    int32_t noise_perlin;
    float noise_scale, px, py, pz;
};
__device__ __forceinline__ void apply_albedo(PathColor& pc, const Albedo& al) {
    if (al.emissive) {
        pc.rad_r += pc.thr_r * al.r; pc.rad_g += pc.thr_g * al.g; pc.rad_b += pc.thr_b * al.b;
    } else {
        pc.thr_r *= al.r; pc.thr_g *= al.g; pc.thr_b *= al.b;
    }
}

template <bool kDeferNoise, bool kPerlinShared = false>
__device__ __forceinline__ bool shade_hit(const SceneView& sc, const float* __restrict__ background, int32_t max_depth, RayD& ray,
                                          const Best& best, const Sampler& smp, PathColor& pc, int& bounce, Albedo& al) {
    bool end_path = false;
    al.r = al.g = al.b = 1.f;
    al.emissive = false;
    al.noise_perlin = -1;
    al.noise_scale = al.px = al.py = al.pz = 0.f;
    if (best.rec < 0) {  // background (Q8)
        pc.rad_r += pc.thr_r * background[0]; pc.rad_g += pc.thr_g * background[1]; pc.rad_b += pc.thr_b * background[2];
        end_path = true;
    } else {
        HitOut ho;
        finalize_hit<false>(sc, ray, best, ho);
        int32_t mkind, mtex;
        float alb_r = 0.f, alb_g = 0.f, alb_b = 0.f, mparam = 0.f;
        if (ho.material < 0) {  // ConstantMedium's own Isotropic (hittable.rs:726,786)
            mkind = RTX_MAT_ISOTROPIC;
            mtex = -(ho.material + 1);
        } else {
            DMaterial m = sc.materials[ho.material];
            mkind = m.kind; mtex = m.texture; alb_r = m.albedo[0]; alb_g = m.albedo[1]; alb_b = m.albedo[2]; mparam = m.param;
        }
        // Texture::value for the three materials that carry one (material.rs:97,247,262)
        if (mkind == RTX_MAT_LAMBERTIAN || mkind == RTX_MAT_ISOTROPIC || mkind == RTX_MAT_DIFFUSE_LIGHT) {
            float tu = 0.f, tv = 0.f;  // (moving spheres and media: u = v = 0, Q10 / Q16)
            if (sc.textures[mtex]._pad) {  // only image lookups need the surface coordinates
                if (ho.type == REC_SPHERE) {  // Sphere::uv (hittable.rs:77-83) in fp32
                    const float PI = 3.14159265358979f;
                    tv = acosf(-(float)ho.on.y) / PI;
                    tu = (atan2f(-(float)ho.on.z, (float)ho.on.x) + PI) / (2.f * PI);
                } else if (ho.type >= REC_RECT_XY && ho.type <= REC_RECT_YZ) {
                    rect_uv(sc, best.rec, ho.ru, ho.rv, tu, tv);
                }
            }
            DTexture t = resolve_texture(sc, mtex, ho.p);
            if (kDeferNoise && t.kind == RTX_TEX_NOISE) {
                al.noise_perlin = t.a;
                al.noise_scale = t.f[0];
                al.px = (float)ho.p.x; al.py = (float)ho.p.y; al.pz = (float)ho.p.z;
            } else {
                f3 tex = texture_eval<kPerlinShared>(sc, t, tu, tv, ho.p);
                alb_r = tex.x; alb_g = tex.y; alb_b = tex.z;
            }
        }
        if (mkind == RTX_MAT_DIFFUSE_LIGHT) {  // material.rs:242-250 (Q24): emits on both sides, never scatters
            al.emissive = true;
            end_path = true;
        } else {
            // The random draws of scatter(): block (SCATTER, 0) serves every material — words 0..2 are the
            // first candidate of Vec3f::random_in_unit_space (vec3.rs:149-160; Lambertian, Isotropic and
            // Metal keep drawing blocks until one lies in the ball), word 3 the Dielectric's uniform
            // (material.rs:189). The candidates are exact in fp32 and their squared length is exact in f64,
            // so accept / reject decisions are the oracle's.
            const bool ball = mkind != RTX_MAT_DIELECTRIC;
            d3 b;
            uint32_t w3 = 0;
            for (uint32_t j = 0;; ++j) {
                uint4 w = smp.block(P_SCATTER, j);
                if (j == 0) w3 = w.w;
                b = mk(2.0 * u01d(w.x) - 1.0, 2.0 * u01d(w.y) - 1.0, 2.0 * u01d(w.z) - 1.0);
                if (!ball || dot(b, b) < 1.0) break;
            }
            d3 nd;
            if (mkind == RTX_MAT_LAMBERTIAN) {  // material.rs:90-99 (Q2)
                nd = mk(ho.p.x + ho.n.x + b.x - ho.p.x, ho.p.y + ho.n.y + b.y - ho.p.y, ho.p.z + ho.n.z + b.z - ho.p.z);
            } else if (mkind == RTX_MAT_ISOTROPIC) {  // material.rs:256-266 (Q3)
                nd = b;
            } else {
                double k = 1.0 / sqrt(dot(ray.d, ray.d));
                d3 udir = k * ray.d;  // Vec3f::unit of the incoming direction
                d3 refl = udir - (2.0 * dot(udir, ho.n)) * ho.n;
                if (mkind == RTX_MAT_METAL) {  // material.rs:134-148 (Q4)
                    nd = refl + (double)mparam * b;
                    if (!(dot(nd, ho.n) > 0.0)) end_path = true;  // absorbed: only `emitted` (= 0) is returned
                } else {  // RTX_MAT_DIELECTRIC, material.rs:180-203 (Q5, Q6); attenuation (1,1,1)
                    double ir = (double)mparam;
                    double ratio = ho.front_face ? 1.0 / ir : ir;
                    double cos_theta = fmin(dot(-udir, ho.n), 1.0);
                    double sin_theta = sqrt(1.0 - cos_theta * cos_theta);
                    bool reflect = ratio * sin_theta > 1.0;
                    if (!reflect) {
                        double r0 = (1.0 - ratio) / (1.0 + ratio);
                        r0 = r0 * r0;
                        double om = 1.0 - cos_theta;
                        double schlick = r0 + (1.0 - r0) * (om * om * om * om * om);
                        reflect = schlick > u01d(w3);
                    }
                    nd = refl;
                    if (!reflect) {  // vec3.rs:116-121
                        d3 perp = ratio * (udir + cos_theta * ho.n);
                        d3 par = (-sqrt(fabs(1.0 - dot(perp, perp)))) * ho.n;
                        nd = perp + par;
                    }
                    alb_r = alb_g = alb_b = 1.f;
                }
            }
            ray.d = nd;
            ray.o = ho.p;
            ++bounce;
            if (bounce >= max_depth) end_path = true;  // color(depth = 0) returns 0
        }
        al.r = alb_r; al.g = alb_g; al.b = alb_b;  // (a deferred noise value overwrites this grey)
    }
    return end_path;
}

// Pixel jitter (main.rs:212-214) + Camera::ray (camera.rs:63-84, Q25) for pixel column `px`, row `jrow`
// counted from the bottom (main.rs:202-204), sample smp.sample.
__device__ __forceinline__ void camera_ray(const CameraView& cam, int width, int height, int px, int jrow, const Sampler& smp, RayD& ray) {
    // pixel jitter (main.rs:212-214) + Camera::ray (camera.rs:63-84, Q25): block (CAMERA, 0)
    // holds the jitter and the shutter time, blocks (LENS, j) two disk candidates each. The
    // lens draw is skipped for a pinhole: counter-based draws make that invisible.
    double su = 0.0, sv = 0.0, tm = 0.0, lx = 0.0, ly = 0.0;
    for (uint32_t j = 0;; ++j) {
        uint4 w = smp.block(j == 0 ? P_CAMERA : P_LENS, j == 0 ? 0u : j - 1u);
        if (j == 0) {
            su = ((double)px + u01d(w.x)) / (double)width;
            sv = ((double)jrow + u01d(w.y)) / (double)height;
            tm = u01d(w.z);
            if (cam.lens_radius == 0.0) break;
        } else {
            lx = 2.0 * u01d(w.x) - 1.0; ly = 2.0 * u01d(w.y) - 1.0;
            if (lx * lx + ly * ly < 1.0) break;
            lx = 2.0 * u01d(w.z) - 1.0; ly = 2.0 * u01d(w.w) - 1.0;
            if (lx * lx + ly * ly < 1.0) break;
        }
    }
    double rdx = cam.lens_radius * lx, rdy = cam.lens_radius * ly;
    d3 off = mk(cam.u[0] * rdx + cam.v[0] * rdy, cam.u[1] * rdx + cam.v[1] * rdy, cam.u[2] * rdx + cam.v[2] * rdy);
    ray.o = mk(cam.origin[0] + off.x, cam.origin[1] + off.y, cam.origin[2] + off.z);
    ray.d = mk(cam.lower_left[0] + su * cam.horizontal[0] + sv * cam.vertical[0] - cam.origin[0] - off.x,
               cam.lower_left[1] + su * cam.horizontal[1] + sv * cam.vertical[1] - cam.origin[1] - off.y,
               cam.lower_left[2] + su * cam.horizontal[2] + sv * cam.vertical[2] - cam.origin[2] - off.z);
    ray.time = cam.time0 + (cam.time1 - cam.time0) * tm;
}

struct RenderArgs {
    SceneView sc;
    CameraView cam;
    int32_t width, height, spp_begin, spp_count, max_depth;
    uint32_t k0, k1;
    int32_t tiles_x, tiles_y;
    float inv_per_block_row;  // 1 / (tiles_x * kBlockH), see tile_of_order
    // phase scheduling weights (see render_kernel): a phase runs when weight * lanes waiting for it is the largest
    int32_t w_node, w_leaf, w_shade;
    int32_t node_burst;  // node steps per vote, at most
};

constexpr int kTileW = 8, kTileH = 4;  // work tile = 8x4 pixels x spp_count samples

// The order in which the dispenser hands out the tiles of a frame: blocks of kBlockW x kBlockH tiles (32 x 128 pixels),
// the blocks row by row, the tiles inside a block row by row. What is in flight at any time is a run of consecutive
// tiles of this order (512 Ki paths = 128 tiles at 128 spp): in row-major order that run is a strip 800 pixels wide and
// 5 high, here it is one block, so the paths in flight start from the same corner of the scene. Scene 9 showed the effect
// first: its throughput rises with the samples per call — 599 M samples/s at 128 spp, 614 at 512, 638 at 2048, 661 at
// 10 000 — for no other reason than that the tiles in flight get fewer and closer together. Measured on scene 9 at
// 128 / 512 spp against row-major 603 / 617: blocks of 8x16 tiles 621 / 650, 16x32 622 / 644, 4x8 612 / 650,
// 4x16 624 / 653, 4x32 630 / 653, 2x64 630 / 650, 1x128 628 / 642; the Cornell scenes and scene 1 do not care (+-0.5 %).
// (Results do not depend on the order: every random draw is keyed by pixel, sample and bounce.)
#ifndef RTX_BLOCK_W
#define RTX_BLOCK_W 4
#endif
#ifndef RTX_BLOCK_H
#define RTX_BLOCK_H 32
#endif
constexpr int kBlockW = RTX_BLOCK_W, kBlockH = RTX_BLOCK_H;
// inv_per_block_row = 1.0f / (tiles_x * kBlockH), from the host: the one division by a frame-dependent number becomes a
// multiplication and a correction (a 32-bit division is ~25 instructions, and every refill of every warp pays the mapping:
// with four of them the Cornell scenes lost 1-2 %).
__host__ __device__ __forceinline__ void tile_of_order(unsigned int k, int tiles_x, int tiles_y, float inv_per_block_row, int& tx, int& ty) {
    const unsigned int per_block_row = (unsigned int)tiles_x * kBlockH;
    unsigned int br = (unsigned int)((float)k * inv_per_block_row);
    int rem_s = (int)(k - br * per_block_row);
    if (rem_s < 0) { --br; rem_s += (int)per_block_row; }
    else if (rem_s >= (int)per_block_row) { ++br; rem_s -= (int)per_block_row; }
    const unsigned int rem = (unsigned int)rem_s;
    const int bh = min(kBlockH, tiles_y - (int)br * kBlockH);      // (the last block row may be lower)
    unsigned int bc, r2;
    if (bh == kBlockH) { bc = rem / (unsigned int)(kBlockW * kBlockH); r2 = rem % (unsigned int)(kBlockW * kBlockH); }  // (shifts)
    else { bc = rem / (unsigned int)(kBlockW * bh); r2 = rem - bc * (unsigned int)(kBlockW * bh); }
    const int bw = min(kBlockW, tiles_x - (int)bc * kBlockW);      // (the last block of a row may be narrower)
    unsigned int q, m;
    if (bw == kBlockW) { q = r2 / (unsigned int)kBlockW; m = r2 % (unsigned int)kBlockW; }
    else { q = r2 / (unsigned int)bw; m = r2 - q * (unsigned int)bw; }
    ty = (int)br * kBlockH + (int)q;
    tx = (int)bc * kBlockW + (int)m;
}
// (the inverse; tools/tile_order_check.cu and tests/test_host_cpu.py check the pair on ragged and very large grids)
__host__ __device__ __forceinline__ unsigned int order_of_tile(int tx, int ty, int tiles_x, int tiles_y) {
    const int br = ty / kBlockH, bc = tx / kBlockW;
    const int bh = min(kBlockH, tiles_y - br * kBlockH), bw = min(kBlockW, tiles_x - bc * kBlockW);
    return (unsigned int)(br * tiles_x * kBlockH + bc * kBlockW * bh + (ty - br * kBlockH) * bw + (tx - bc * kBlockW));
}
constexpr int kRenderBlock = 128;

enum LaneState : int32_t {
    ST_NEW = 0,    // needs a path sample from the pool
    ST_TRAV = 1,   // has a ray in flight
    ST_SHADE = 2,  // closest hit known, waiting for the shade phase
    ST_DONE = 3    // pool empty, nothing left for this lane
};

// ---------------------------------------------------------------------------
// K2: the path loop (render()'s pixel loop + color(), main.rs:26-45,202-217).
//
// A warp is the scheduling unit. Its 32 lanes each carry one path; a lane that finishes a path
// takes the next (pixel, sample) item from the warp's pool (an 8x4 pixel tile x spp_count
// samples, refilled from a global tile counter), so no lane waits for a neighbour's longer
// path. The work of a path step comes in three kinds with very different code — BVH node steps
// (fp32), leaf events (f64 primitive tests) and shading (hit
// record, material, texture, Philox, next ray, medium pre-pass) — and lanes reach them at
// different times. Instead of letting every lane run its own branch (the first version of this
// kernel: 7 of 32 lanes active on average), the warp votes each iteration and runs ONE phase for
// all lanes that are waiting for it: the phase with the most (weighted) waiting lanes. Lanes that
// reach a leaf keep traversing speculatively with the leaf postponed (they block on the second).
// ---------------------------------------------------------------------------
template <bool kCount>
__global__ void __launch_bounds__(kRenderBlock) render_kernel(RenderArgs a, float4* __restrict__ accum, unsigned long long* ray_count,
                                                              unsigned int* work_counter, Counters* counters) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const uint32_t lt_mask = (1u << lane) - 1u;
    int32_t stack[kStackSize];
    Tally<kCount> tally;
    const uint32_t n_tiles = (uint32_t)(a.tiles_x * a.tiles_y);
    const float tmin_f = __double2float_rd(0.001);
    // the warp's pool of path samples (warp-uniform)
    uint32_t pool_next = 0, pool_end = 0;
    int pool_x0 = 0, pool_y0 = 0;
    bool pool_dry = false;
    // lane state
    int32_t st = ST_NEW;
    RayD ray{mk(0, 0, 0), mk(0, 0, 1), 0.0};
    SlabRay sr{0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    Best best{0.0, -1, 0};
    float tmax_f = 0.f;
    int32_t cur = kSentinel, pending = 0;  // pending: a postponed leaf (leaf codes are negative; 0 = none)
    int sp = 0;
    Sampler smp{a.k0, a.k1, 0u, 0u, 0u};
    PathColor pc{1.f, 1.f, 1.f, 0.f, 0.f, 0.f};
    int bounce = 0;
    unsigned long long my_rays = 0;

    while (true) {
        // ---- cheap per-lane transitions, then the vote ----
        if (st == ST_TRAV && cur < 0) {
            if (cur == kSentinel) {
                if (pending == 0) st = ST_SHADE;
            } else if (pending == 0) {
                pending = cur;  // postpone the leaf, keep traversing (speculatively: best.t is not shrunk yet)
                cur = stack[--sp];
            }
        }
        const bool want_node = st == ST_TRAV && cur >= 0;
        const bool want_leaf = st == ST_TRAV && cur < 0 && pending != 0;
        const bool want_shade = st == ST_SHADE || st == ST_NEW;
        const int n_node = __popc(__ballot_sync(FULL, want_node));
        const int n_leaf = __popc(__ballot_sync(FULL, want_leaf));
        const int n_shade = __popc(__ballot_sync(FULL, want_shade));
        if ((n_node | n_leaf | n_shade) == 0) {
            // lanes that popped a leaf / sentinel this very iteration settle on the next one; only ST_DONE ends the loop
            if (__all_sync(FULL, st == ST_DONE)) break;
            continue;
        }
        const int s_node = n_node * a.w_node, s_leaf = n_leaf * a.w_leaf, s_shade = n_shade * a.w_shade;

        if (s_node >= s_leaf && s_node >= s_shade) {
            // ================= node phase =================
            // a burst of node steps: stay while at least half of the lanes that started it still have a node
            bool go = want_node;
#pragma unroll 1
            for (int it = 0; it < a.node_burst; ++it) {
                if (go) {
                    cur = node_step(a.sc, cur, sr, tmin_f, tmax_f, stack, sp, tally);
                    if (cur < 0 && cur != kSentinel && pending == 0) {
                        pending = cur;  // postpone the leaf, keep traversing
                        cur = stack[--sp];
                    }
                    go = cur >= 0;
                }
                if (2 * __popc(__ballot_sync(FULL, go)) < n_node) break;
            }
        } else if (s_leaf >= s_shade) {
            // ================= leaf phase =================
            if (want_leaf) {
                int32_t v = ~pending;
                int32_t first = v >> 4, count = v & 15;
                pending = 0;
                for (int32_t i = 0; i < count; ++i) {
                    int4 h = __ldg(reinterpret_cast<const int4*>(a.sc.records + first + i));
                    double t;
                    int32_t hit_rec;
                    if (test_geometry(a.sc, first + i, h, ray, 0.001, best.t, t, hit_rec, tally)) {
                        best.t = t;
                        best.rec = hit_rec;
                        best.chain = h.w;
                        tmax_f = __double2float_ru(t);
                    }
                }
            }
        } else {
            // ================= shade phase =================
            bool fresh = false;  // this lane leaves the phase with a new ray to trace
            if (st == ST_SHADE) {
                Albedo al;
                const bool end_path = shade_hit<false>(a.sc, a.cam.background, a.max_depth, ray, best, smp, pc, bounce, al);
                apply_albedo(pc, al);
                if (end_path) {
                    // one path sample done: add it to its pixel (sum r, g, b, count)
                    atomicAdd(accum + smp.pixel, make_float4(pc.rad_r, pc.rad_g, pc.rad_b, 1.0f));
                    st = ST_NEW;
                } else {
                    fresh = true;
                }
            }
            // ---- hand out path samples to the lanes that need one ----
            uint32_t need = __ballot_sync(FULL, st == ST_NEW);
            while (need != 0) {
                if (pool_next >= pool_end) {  // warp-uniform: refill from the global tile counter
                    if (!pool_dry) {
                        unsigned int tile = 0;
                        if (lane == 0) tile = atomicAdd(work_counter, 1u);
                        tile = __shfl_sync(FULL, tile, 0);
                        if (tile < n_tiles) {
                            int tx, ty;
                            tile_of_order(tile, a.tiles_x, a.tiles_y, a.inv_per_block_row, tx, ty);
                            pool_x0 = tx * kTileW;
                            pool_y0 = ty * kTileH;
                            pool_next = 0;
                            pool_end = 32u * (uint32_t)a.spp_count;
                        } else {
                            pool_dry = true;
                        }
                    }
                    if (pool_dry) {
                        if (st == ST_NEW) st = ST_DONE;
                        break;
                    }
                }
                const uint32_t avail = pool_end - pool_next;
                const uint32_t rank = (uint32_t)__popc(need & lt_mask);
                const bool take = ((need >> lane) & 1u) != 0 && rank < avail;
                if (take) {
                    // item -> (sample, pixel of the tile): consecutive items are the 32 pixels of one sample index
                    const uint32_t item = pool_next + rank;
                    const int pi = (int)(item & 31u);
                    const int px = pool_x0 + (pi & (kTileW - 1)), row = pool_y0 + (pi / kTileW);  // row 0 = top
                    if (px < a.width && row < a.height) {
                        const int jrow = a.height - 1 - row;  // main.rs:202-204: j runs height-1 .. 0, top row first
                        smp.pixel = (uint32_t)(row * a.width + px);
                        smp.sample = (uint32_t)a.spp_begin + (item >> 5);
                        smp.bounce = 0;
                        if (a.max_depth <= 0) {  // color(.., depth = 0) is black without tracing anything (main.rs:27-29)
                            atomicAdd(accum + smp.pixel, make_float4(0.f, 0.f, 0.f, 1.0f));
                        } else {
                            camera_ray(a.cam, a.width, a.height, px, jrow, smp, ray);
                            pc = PathColor{1.f, 1.f, 1.f, 0.f, 0.f, 0.f};
                            bounce = 0;
                            fresh = true;
                            st = ST_TRAV;
                        }
                    }
                    // (a pixel outside a ragged image edge, or depth 0: the lane stays ST_NEW and takes another item)
                }
                pool_next += min((uint32_t)__popc(need), avail);
                need = __ballot_sync(FULL, st == ST_NEW);
            }
            // ---- new rays: media first, then the surface traversal starts at the world root ----
            if (fresh) {
                smp.bounce = (uint32_t)bounce;
                best.t = 1.7976931348623157e308;
                best.rec = -1;
                best.chain = 0;
                make_slab(ray.o, ray.d, sr);
                if (a.sc.n_media > 0) media_prepass<false>(a.sc, ray, sr, 0.001, best, 0.0, &smp, stack, tally);
                tmax_f = __double2float_ru(best.t);
                sp = 0;
                stack[sp++] = kSentinel;
                cur = a.sc.world_root;
                pending = 0;
                st = ST_TRAV;
                ++my_rays;
            }
        }
    }
    if (ray_count) {
        for (int off = 16; off > 0; off >>= 1) my_rays += __shfl_xor_sync(FULL, my_rays, off);
        if (lane == 0 && my_rays) atomicAdd(ray_count, my_rays);
    }
    if constexpr (kCount) {
        uint32_t vals[4] = {tally.n_node, tally.n_sphere, tally.n_rect, tally.n_med};
#pragma unroll
        for (int k = 0; k < 4; ++k)
            for (int off = 16; off > 0; off >>= 1) vals[k] += __shfl_xor_sync(FULL, vals[k], off);
        if (lane == 0) {
            atomicAdd(&counters->node_visits, (unsigned long long)vals[0]);
            atomicAdd(&counters->box_tests, 2ull * vals[0]);
            atomicAdd(&counters->sphere_tests, (unsigned long long)vals[1]);
            atomicAdd(&counters->rect_tests, (unsigned long long)vals[2]);
            atomicAdd(&counters->medium_tests, (unsigned long long)vals[3]);
        }
    }
}

// ---------------------------------------------------------------------------
// K2w: the same path loop as a WAVEFRONT. Paths live in a pool of slots in HBM (SoA, 96 bytes per
// slot, L2-resident at the default pool size); one iteration = wf_shade_kernel (every slot: shade
// the hit found for its ray, scatter or end the path, refill empty slots with new camera rays, run
// the medium pre-pass for the new ray) followed by wf_trace_kernel (every slot: closest surface
// hit of its ray). Each kernel then has ONE kind of work per thread, which is what the
// megakernel's warp votes try to recover; the price is the pool traffic (~300 B per ray).
// ---------------------------------------------------------------------------
struct PathPool {
    double *ox, *oy, *oz, *dx, *dy, *dz, *time, *best_t;
    int32_t *best_rec, *best_chain, *bounce;  // bounce < 0: empty slot
    uint32_t *pixel, *sample;
    float *thr_r, *thr_g, *thr_b;  // (no radiance: every emission ends its path — DiffuseLight never scatters, the background is a miss — so a path in flight has gathered none yet)
};
constexpr int kPoolBytesPerSlot = 8 * 8 + 8 * 4;

struct AdaptiveArgs {
    const uint32_t* tile_list;  // dispenser tile k renders tile_of_order(tile_list[k], ...)
    float4* aux;                // receives the samples with an odd global index a second time
};

struct WfArgs {
    SceneView sc;
    CameraView cam;
    PathPool pool;
    int32_t width, height, spp_begin, spp_count, max_depth;
    uint32_t k0, k1;
    int32_t tiles_x, tiles_y;
    float inv_per_block_row;  // 1 / (tiles_x * kBlockH), see tile_of_order
    int32_t n_slots;
    unsigned long long total_items;   // tiles * 32 * spp_count
    unsigned long long* next_item;    // global dispenser of path samples
    // Last, what one specialisation of the shade kernel needs, never both: ray ordering for the trace pass (order.cuh,
    // kOrder) or adaptive sampling (adaptive.cuh, kAdaptive). Sharing the space keeps the size of WfArgs, so the kernel
    // parameters behind it, and the code of every other shade kernel, stay where they were.
    union {
        OrderArgs order;
        AdaptiveArgs adaptive;
    };
};

constexpr int kWfBlock = 128;   // trace kernel CTA; the pool size is a multiple of it
#ifndef WF_SHADE_BLOCK
#define WF_SHADE_BLOCK 128
#endif
constexpr int kShadeBlock = WF_SHADE_BLOCK;  // shade kernel CTA (divides kWfBlock)
#ifndef WF_TRACE_BLOCK
#define WF_TRACE_BLOCK 128
#endif
constexpr int kTraceBlock = WF_TRACE_BLOCK;  // trace kernel CTA (divides kWfBlock): registers are released per CTA
#ifndef WF_TRACE_MINB
#define WF_TRACE_MINB 7
#endif
#ifndef WF_SHADE_MINB
#define WF_SHADE_MINB 5
#endif

// One pass: shade the hit of the slot (one level of color()), add a finished path's sample to the image, refill
// emptied slots per warp (one dispenser atomic per warp; 32 consecutive items = the pixels of one 8x4 tile at one
// sample index), run the medium pre-pass for the new ray and write the slot. A three-pass variant that generated
// the camera rays densely through shared memory was measured and dropped (DESIGN.md §4: the barriers cost more
// than the dense generation saves, except on the Cornell box).
template <bool kCount>
__global__ void __launch_bounds__(kShadeBlock, WF_SHADE_MINB * (128 / kShadeBlock)) wf_shade_kernel(WfArgs a, float4* __restrict__ accum, unsigned int* active_out, Counters* counters) {
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int i = blockIdx.x * blockDim.x + tid;
    const bool valid = i < a.n_slots;
    int32_t stack[kStackSize];  // only a ConstantMedium with a general boundary traverses here
    Tally<kCount> tally;

    // ---- pass 1: shade ----
    int bounce = valid ? a.pool.bounce[i] : -2;
    RayD ray{mk(0, 0, 0), mk(0, 0, 1), 0.0};
    PathColor pc{1.f, 1.f, 1.f, 0.f, 0.f, 0.f};
    Sampler smp{a.k0, a.k1, 0u, 0u, 0u};
    bool fresh = false, shaded = false, ended = false;
    Albedo al;
    al.noise_perlin = -1;
    if (bounce >= 0) {
        ray.o = mk(a.pool.ox[i], a.pool.oy[i], a.pool.oz[i]);
        ray.d = mk(a.pool.dx[i], a.pool.dy[i], a.pool.dz[i]);
        ray.time = a.pool.time[i];
        Best best{a.pool.best_t[i], a.pool.best_rec[i], a.pool.best_chain[i]};
        pc = PathColor{a.pool.thr_r[i], a.pool.thr_g[i], a.pool.thr_b[i], 0.f, 0.f, 0.f};
        smp.pixel = a.pool.pixel[i];
        smp.sample = a.pool.sample[i];
        smp.bounce = (uint32_t)bounce;
        // (a dense shared-memory pass for Perlin textures — shade_hit<true> + noise_value for queued threads — was
        // measured: neutral on scenes 3 / 5, -2 % on scene 9 for its two extra barriers; not used)
        ended = shade_hit<false>(a.sc, a.cam.background, a.max_depth, ray, best, smp, pc, bounce, al);
        shaded = true;
    }
    if (shaded) {
        apply_albedo(pc, al);
        if (ended) {
            atomicAdd(accum + smp.pixel, make_float4(pc.rad_r, pc.rad_g, pc.rad_b, 1.0f));  // one path sample done
            bounce = -1;
            a.pool.bounce[i] = -1;
        } else {
            fresh = true;
        }
    }
    {   // ---- refill empty slots per warp: consecutive items are the 32 pixels of one tile at one sample index ----
        const bool want = bounce == -1;
        unsigned m = __ballot_sync(FULL, want);
        if (m != 0 && __ldcg(a.next_item) >= a.total_items) m = 0;  // dispenser already dry: no atomic
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
                tile_of_order(tile, a.tiles_x, a.tiles_y, a.inv_per_block_row, tx, ty);
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

    // ---- pass 3: the new ray: media first (their scatter point bounds the surface search), then out to the pool ----
    if (fresh) {
        smp.bounce = (uint32_t)bounce;
        Best best{1.7976931348623157e308, -1, 0};
        if (a.sc.n_media > 0) {
            SlabRay sr;
            make_slab(ray.o, ray.d, sr);
            media_prepass<false>(a.sc, ray, sr, 0.001, best, 0.0, &smp, stack, tally);
        }
        a.pool.ox[i] = ray.o.x; a.pool.oy[i] = ray.o.y; a.pool.oz[i] = ray.o.z;
        a.pool.dx[i] = ray.d.x; a.pool.dy[i] = ray.d.y; a.pool.dz[i] = ray.d.z;
        a.pool.time[i] = ray.time;
        a.pool.best_t[i] = best.t; a.pool.best_rec[i] = best.rec; a.pool.best_chain[i] = best.chain;
        a.pool.thr_r[i] = pc.thr_r; a.pool.thr_g[i] = pc.thr_g; a.pool.thr_b[i] = pc.thr_b;
        a.pool.pixel[i] = smp.pixel; a.pool.sample[i] = smp.sample;
        a.pool.bounce[i] = bounce;
    }
    if (active_out) {
        const unsigned am = __ballot_sync(FULL, fresh);
        if (lane == 0 && am != 0) atomicAdd(active_out, (unsigned int)__popc(am));
    }
    if constexpr (kCount) {
        uint32_t v = tally.n_med;
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(FULL, v, off);
        if (lane == 0 && v) atomicAdd(&counters->medium_tests, (unsigned long long)v);
        // (node / primitive counts of general medium boundaries are not attributed)
    }
}

template <bool kCount, bool kWide = false>
__global__ void __launch_bounds__(kTraceBlock, WF_TRACE_MINB * (128 / kTraceBlock)) wf_trace_kernel(SceneView sc, PathPool pool, int n_slots, unsigned long long* ray_count,
                                                            Counters* counters) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int32_t stack[kStackSize];
    Tally<kCount> tally;
    const bool act = i < n_slots && pool.bounce[i] >= 0;
    if (act) {
        RayD ray{mk(pool.ox[i], pool.oy[i], pool.oz[i]), mk(pool.dx[i], pool.dy[i], pool.dz[i]), pool.time[i]};
        Best best{pool.best_t[i], -1, 0};
        if constexpr (kWide) traverse_wide(sc, sc.wide_root, ray, 0.001, best, stack, tally);
        else traverse_simple(sc, sc.world_root, ray, 0.001, best, stack, 0, tally);
        if (best.rec >= 0) {  // closer than the medium candidate (if any) the shade kernel left there
            pool.best_t[i] = best.t;
            pool.best_rec[i] = best.rec;
            pool.best_chain[i] = best.chain;
        }
    }
    if (ray_count) {
        const unsigned am = __ballot_sync(FULL, act);
        if (lane == 0 && am != 0) atomicAdd(ray_count, (unsigned long long)__popc(am));
    }
    if constexpr (kCount) {
        uint32_t vals[3] = {tally.n_node, tally.n_sphere, tally.n_rect};
#pragma unroll
        for (int k = 0; k < 3; ++k)
            for (int off = 16; off > 0; off >>= 1) vals[k] += __shfl_xor_sync(FULL, vals[k], off);
        if (lane == 0) {
            atomicAdd(&counters->node_visits, (unsigned long long)vals[0]);
            atomicAdd(&counters->box_tests, 2ull * vals[0]);
            atomicAdd(&counters->sphere_tests, (unsigned long long)vals[1]);
            atomicAdd(&counters->rect_tests, (unsigned long long)vals[2]);
        }
    }
}

// The same kernel taking its rays in the order the shade pass and wf_order_kernel prepared (order.cuh): thread p traces the
// ray of slot order[p]. Threads past the number of rays in flight have nothing to do.
template <bool kCount>
__global__ void __launch_bounds__(kTraceBlock, WF_TRACE_MINB * (128 / kTraceBlock)) wf_trace_ordered_kernel(SceneView sc, PathPool pool, OrderArgs o, unsigned long long* ray_count,
                                                                                                              Counters* counters) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n_live = __ldg(o.offsets + o.n_bins_padded);
    const uint32_t i = __ldg(o.order + p);  // (in bounds for every thread of the launch; meaningful for p < n_live)
    if (ray_count && p == 0) atomicAdd(ray_count, (unsigned long long)n_live);
    if (blockIdx.x * blockDim.x >= n_live) return;
    int32_t stack[kStackSize];
    Tally<kCount> tally;
    if (p < n_live) {
        RayD ray{mk(pool.ox[i], pool.oy[i], pool.oz[i]), mk(pool.dx[i], pool.dy[i], pool.dz[i]), pool.time[i]};
        Best best{pool.best_t[i], -1, 0};
        traverse_simple(sc, sc.world_root, ray, 0.001, best, stack, 0, tally);
        if (best.rec >= 0) {
            pool.best_t[i] = best.t;
            pool.best_rec[i] = best.rec;
            pool.best_chain[i] = best.chain;
        }
    }
    if constexpr (kCount) {
        uint32_t vals[3] = {tally.n_node, tally.n_sphere, tally.n_rect};
#pragma unroll
        for (int k = 0; k < 3; ++k)
            for (int off = 16; off > 0; off >>= 1) vals[k] += __shfl_xor_sync(FULL, vals[k], off);
        if (lane == 0) {
            atomicAdd(&counters->node_visits, (unsigned long long)vals[0]);
            atomicAdd(&counters->box_tests, 2ull * vals[0]);
            atomicAdd(&counters->sphere_tests, (unsigned long long)vals[1]);
            atomicAdd(&counters->rect_tests, (unsigned long long)vals[2]);
        }
    }
}

// (Two persistent forms of the trace kernel — warp-voted node / leaf / fetch phases, and refill at the top
// of a while-while loop — were measured in round 1 at equal registers and lost to the form above:
// 365 M and 400 M vs 413 M path samples/s on scene 9. DESIGN.md §4 has the numbers; the code is in the
// history, commit "Wavefront defaults ...".)

// color(.., depth = 0) is black without tracing anything (main.rs:27-29): count the samples only
__global__ void add_black_samples_kernel(float4* __restrict__ accum, int n_pixels, float count) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_pixels) accum[i].w += count;
}

// ---------------------------------------------------------------------------
// K3: main.rs:217-225 (Q26). NaN -> 0 like Rust's `as u8`.
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint8_t quantise(float sum, float inv_n) {
    float x = sqrtf(sum * inv_n);
    x = fminf(fmaxf(x, 0.f), 0.999f) * 256.f;  // fmaxf/fminf drop NaN -> 0
    return (uint8_t)(int)x;
}
__global__ void tonemap_kernel(const float4* __restrict__ accum, int n_pixels, uchar4* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pixels) return;
    float4 a = accum[i];
    float inv = 1.0f / a.w;
    out[i] = make_uchar4(quantise(a.x, inv), quantise(a.y, inv), quantise(a.z, inv), 255);
}

constexpr int kMaxPeers = 16;
struct PeerList {
    const float4* p[kMaxPeers];
    int n;
};
// Rank-0 side of the multi-GPU combine: reads every peer's accumulator straight over NVLink
// (peer-mapped pointers), adds it to the local one, writes the sum back and tonemaps — one pass.
__global__ void reduce_tonemap_peers_kernel(float4* __restrict__ accum, PeerList peers, int n_pixels, uchar4* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pixels) return;
    float4 a = accum[i];
    for (int k = 0; k < peers.n; ++k) {
        float4 b = peers.p[k][i];
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    accum[i] = a;
    float inv = 1.0f / a.w;
    out[i] = make_uchar4(quantise(a.x, inv), quantise(a.y, inv), quantise(a.z, inv), 255);
}

// The same combine spread over the ranks: this rank's slice of the pixels, every rank's accumulator read (its own
// locally, the others over NVLink), the RGBA8 result written straight into rank 0's frame. Nothing written back.
__global__ void reduce_tonemap_slice_kernel(PeerList all, int first, int count, uchar4* __restrict__ out_root) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    i += first;
    float4 a = all.p[0][i];
    for (int k = 1; k < all.n; ++k) {
        float4 b = all.p[k][i];
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    float inv = 1.0f / a.w;
    out_root[i] = make_uchar4(quantise(a.x, inv), quantise(a.y, inv), quantise(a.z, inv), 255);
}

// ---------------------------------------------------------------------------
// Measurement aid (rtx_ctx_measure_l2_read): every thread streams 16-byte words of a buffer that fits in L2,
// `repeats` times over, with loads that bypass L1 (ld.global.cg). Four independent loads in flight per thread.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) l2_read_kernel(const uint4* __restrict__ buf, unsigned long long n_vec, int repeats,
                                                      unsigned int* __restrict__ sink) {
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    const unsigned long long first = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned int acc = 0;
    for (int r = 0; r < repeats; ++r) {
        unsigned long long i = first;
        for (; i + 3 * stride < n_vec; i += 4 * stride) {
            const uint4 a = __ldcg(buf + i), b = __ldcg(buf + i + stride), c = __ldcg(buf + i + 2 * stride), d = __ldcg(buf + i + 3 * stride);
            acc ^= a.x ^ a.y ^ a.z ^ a.w ^ b.x ^ b.y ^ b.z ^ b.w ^ c.x ^ c.y ^ c.z ^ c.w ^ d.x ^ d.y ^ d.z ^ d.w;
        }
        for (; i < n_vec; i += stride) {
            const uint4 a = __ldcg(buf + i);
            acc ^= a.x ^ a.y ^ a.z ^ a.w;
        }
        acc = acc * 2654435761u + (unsigned int)r;  // keeps the passes from being merged
    }
    if (acc == 0x9e3779b9u) atomicAdd(sink, 1u);  // practically never; keeps the loads alive
}

}  // namespace rtx
