// oracle_first_vertex.cpp — the feature buffers of rtx_render_aov restated in f64 on the CPU oracle. TEST INFRASTRUCTURE
// ONLY: tests/test_gpu_aov.py compiles it, with the oracle's own flags, into a library of its own. It includes the oracle
// unchanged, so the first vertex is the one orc_render's bounce 0 reaches: the same camera ray, the same world.hit with
// the same Philox draws (each ConstantMedium's free flight), then `emitted` and `scatter` of that vertex.
#include "../oracle/oracle.cpp"

namespace {

// The phase functions of the world's ConstantMedia: a vertex whose material is one of them is a medium scatter point.
void collect_phases(const Hittable* h, std::vector<const Material*>& out) {
    if (!h) return;
    if (auto l = dynamic_cast<const List*>(h)) {
        for (const auto& c : l->list) collect_phases(c.get(), out);
    } else if (auto b = dynamic_cast<const BvhTree*>(h)) {
        collect_phases(b->left.get(), out);
        if (b->right != b->left) collect_phases(b->right.get(), out);
    } else if (auto bl = dynamic_cast<const BvhOfList*>(h)) {
        collect_phases(bl->tree.get(), out);
    } else if (auto t = dynamic_cast<const Translate*>(h)) {
        collect_phases(t->item.get(), out);
    } else if (auto r = dynamic_cast<const YRotate*>(h)) {
        collect_phases(r->item.get(), out);
    } else if (auto m = dynamic_cast<const ConstantMedium*>(h)) {
        out.push_back(&m->phase);
    }
}

Vec3 clamp01(const Vec3& c) {
    return Vec3(std::fmin(std::fmax(c.x, 0.0), 1.0), std::fmin(std::fmax(c.y, 0.0), 1.0), std::fmin(std::fmax(c.z, 0.0), 1.0));
}

}  // namespace

// Adds per pixel (row 0 = top): albedo_sum (width*height*3: the attenuation scatter() returns — Metal's albedo also when
// the scatter is absorbed, (1, 1, 1) for a Dielectric — for a DiffuseLight its emission and for a miss the background,
// both clamped to [0, 1]), normal_sum (width*height*3: the hit record's normal; nothing for a medium vertex or a miss)
// and depth_sum (width*height*2: t * |d|, number of vertices). When spp_count == 1 and kind != NULL,
// kind[pixel] = vertex | material << 2 | fragile << 7 with vertex 0 = miss, 1 = surface, 2 = medium, material an
// rtx_material_kind (0 for a miss) and fragile as orc_trace_rays reports it for that query. Returns the world.hit queries.
extern "C" uint64_t orc_first_vertex(const orc_scene* s, int width, int height, int spp_begin, int spp_count, uint64_t seed,
                                     double* albedo_sum, double* normal_sum, double* depth_sum, uint8_t* kind, int n_threads) {
    Camera camera(s->camera);
    std::vector<const Material*> phases;
    collect_phases(s->world.get(), phases);
    std::atomic<uint64_t> total_rays{0};
    run_parallel(n_threads, height, 1, [&](int64_t b, int64_t e) {
        g_sampler = Sampler();
        g_sampler.fixed = false;
        g_sampler.key[0] = (uint32_t)seed;
        g_sampler.key[1] = (uint32_t)(seed >> 32);
        g_probe.on = kind != nullptr;
        for (int64_t r = b; r < e; ++r) {
            const int j = height - 1 - (int)r;
            for (int i = 0; i < width; ++i) {
                const size_t px = (size_t)r * width + i;
                g_sampler.pixel = (uint32_t)px;
                Vec3 al, nn;
                double dist = 0.0, hits = 0.0;
                for (int sidx = spp_begin; sidx < spp_begin + spp_count; ++sidx) {  // orc_render's pixel loop, bounce 0 only
                    g_sampler.sample = (uint32_t)sidx;
                    g_sampler.bounce = 0;
                    uint32_t w[4];
                    g_sampler.block(P_CAMERA, 0, w);
                    Ray ray = camera.ray(((double)i + u01(w[0])) / (double)width, ((double)j + u01(w[1])) / (double)height);
                    g_sampler.rays++;
                    g_probe.fragile = false;
                    g_probe.nested = 0;
                    g_probe.min_t = INFINITY;
                    HitRecord rec;
                    int k = 0;  // a miss
                    bool fragile;
                    if (s->world->hit(ray, 0.001, DBL_MAX, rec)) {
                        fragile = g_probe.fragile && !(g_probe.min_t > rec.t + 1e-9 * std::fmax(1.0, std::fabs(rec.t)));
                        const Material* m = rec.material;
                        const Vec3 emitted = m->emitted(rec.u, rec.v, rec.p);
                        Vec3 att;
                        Ray scattered;
                        m->scatter(ray, rec, att, scattered);
                        int mk;
                        if (dynamic_cast<const DiffuseLight*>(m)) { mk = RTX_MAT_DIFFUSE_LIGHT; att = clamp01(emitted); }
                        else if (dynamic_cast<const Lambertian*>(m)) mk = RTX_MAT_LAMBERTIAN;
                        else if (dynamic_cast<const Metal*>(m)) mk = RTX_MAT_METAL;
                        else if (dynamic_cast<const Dielectric*>(m)) mk = RTX_MAT_DIELECTRIC;
                        else mk = RTX_MAT_ISOTROPIC;
                        const bool medium = std::find(phases.begin(), phases.end(), m) != phases.end();
                        k = (medium ? 2 : 1) | (mk << 2);
                        al = al + att;
                        if (!medium) nn = nn + rec.normal;
                        dist += rec.t * ray.b.magnitude();
                        hits += 1.0;
                    } else {
                        fragile = g_probe.fragile;
                        al = al + clamp01(s->background);
                    }
                    if (kind && spp_count == 1) kind[px] = (uint8_t)(k | (fragile ? 0x80 : 0));
                }
                if (albedo_sum) { double* p = albedo_sum + 3 * px; p[0] += al.x; p[1] += al.y; p[2] += al.z; }
                if (normal_sum) { double* p = normal_sum + 3 * px; p[0] += nn.x; p[1] += nn.y; p[2] += nn.z; }
                if (depth_sum) { double* p = depth_sum + 2 * px; p[0] += dist; p[1] += hits; }
            }
        }
        g_probe.on = false;
        total_rays += g_sampler.rays;
    });
    return total_rays.load();
}
