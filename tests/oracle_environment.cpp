// oracle_environment.cpp — the environment map of rtx_scene_set_environment restated in f64 on the CPU oracle. TEST
// INFRASTRUCTURE ONLY: tests/test_gpu_environment.py compiles it, with the oracle's own flags, into a library of its own.
// It includes the unchanged oracle (through the first-vertex restatement), keeps each scene's map beside the scene, and
// restates the two loops whose miss reads the background: orc_render's color() and orc_first_vertex's miss albedo.
// The lookup is include/rttnw_b200.h's E(d) with every step in f64: the texel fraction is not rounded to fp32 and
// the two levels of a + f (b - a) and the scale are f64 products of the fp32 texels.
#include "oracle_first_vertex.cpp"

#include <map>
#include <mutex>

namespace {

struct OrcEnv {
    int w = 0, h = 0;
    std::vector<float> rgb;  // w * h * 3, row 0 = top
    double cos_t = 1.0, sin_t = 0.0, scale[3] = {1.0, 1.0, 1.0};
};
std::mutex g_env_mu;
std::map<const orc_scene*, OrcEnv> g_env;

const OrcEnv* env_of(const orc_scene* s) {
    std::lock_guard<std::mutex> lock(g_env_mu);
    auto it = g_env.find(s);
    return it == g_env.end() ? nullptr : &it->second;
}

Vec3 env_value(const OrcEnv& e, const Vec3& d) {
    const double xr = e.cos_t * d.x - e.sin_t * d.z, zr = e.sin_t * d.x + e.cos_t * d.z;
    const double u = 0.5 + std::atan2(xr, -zr) / (2.0 * 3.14159265358979323846);
    const double v = std::atan2(std::hypot(xr, zr), d.y) / 3.14159265358979323846;
    const double X = u * e.w - 0.5, Y = v * e.h - 0.5;
    const double xf = std::floor(X), yf = std::floor(Y), fx = X - xf, fy = Y - yf;
    const int ix = (int)std::fmax(std::fmin(xf, (double)(e.w - 1)), -1.0), iy = (int)std::fmax(std::fmin(yf, (double)(e.h - 1)), -1.0);
    const int i0 = ix < 0 ? e.w - 1 : ix, i1 = ix + 1 >= e.w ? 0 : ix + 1;
    const int j0 = iy < 0 ? 0 : iy, j1 = iy + 1 >= e.h ? e.h - 1 : iy + 1;
    double out[3];
    for (int c = 0; c < 3; ++c) {
        auto t = [&](int i, int j) { return (double)e.rgb[3 * ((size_t)j * e.w + i) + c]; };
        const double a = t(i0, j0) + fx * (t(i1, j0) - t(i0, j0)), b = t(i0, j1) + fx * (t(i1, j1) - t(i0, j1));
        out[c] = (a + fy * (b - a)) * e.scale[c];
    }
    return Vec3(out[0], out[1], out[2]);
}

Vec3 miss_value(const orc_scene* s, const OrcEnv* e, const Ray& ray) { return e ? env_value(*e, ray.b) : s->background; }

// color() of oracle.cpp (main.rs:26-45) with the miss reading the map
Vec3 color_env(const orc_scene* s, const OrcEnv* e, const Ray& ray, int depth, int max_depth) {
    if (depth <= 0) return Vec3::repeat(0.);
    g_sampler.bounce = (uint32_t)(max_depth - depth);
    g_sampler.rays++;
    HitRecord rec;
    if (s->world->hit(ray, 0.001, DBL_MAX, rec)) {
        Vec3 emitted = rec.material->emitted(rec.u, rec.v, rec.p);
        Vec3 att;
        Ray scattered;
        if (rec.material->scatter(ray, rec, att, scattered)) return emitted + att * color_env(s, e, scattered, depth - 1, max_depth);
        return emitted;
    }
    return miss_value(s, e, ray);
}

}  // namespace

// env == NULL removes the scene's map. Copies the texels.
extern "C" void orc_scene_set_environment(const orc_scene* s, const rtx_environment* env) {
    std::lock_guard<std::mutex> lock(g_env_mu);
    if (!env) { g_env.erase(s); return; }
    OrcEnv e;
    e.w = env->width;
    e.h = env->height;
    e.rgb.assign(env->rgb, env->rgb + (size_t)env->width * env->height * 3);
    const double th = env->rotation_y * (3.14159265358979323846 / 180.0);
    e.cos_t = std::cos(th);
    e.sin_t = std::sin(th);
    for (int c = 0; c < 3; ++c) e.scale[c] = env->scale[c];
    g_env[s] = std::move(e);
}

// E(d) of the scene's map for n directions (the background without a map): rgb is n * 3 doubles.
extern "C" void orc_environment_value(const orc_scene* s, int64_t n, const double* dirs, double* rgb) {
    const OrcEnv* e = env_of(s);
    for (int64_t k = 0; k < n; ++k) {
        Ray r;
        r.b = Vec3(dirs[3 * k], dirs[3 * k + 1], dirs[3 * k + 2]);
        const Vec3 v = miss_value(s, e, r);
        rgb[3 * k] = v.x; rgb[3 * k + 1] = v.y; rgb[3 * k + 2] = v.z;
    }
}

// orc_render (oracle.cpp) with the scene's map.
extern "C" uint64_t orc_render_env(const orc_scene* s, int width, int height, int spp_begin, int spp_count, int max_depth,
                                   uint64_t seed, double* rgb_sum, int n_threads) {
    Camera camera(s->camera);
    const OrcEnv* e = env_of(s);
    std::atomic<uint64_t> total_rays{0};
    run_parallel(n_threads, height, 1, [&](int64_t b, int64_t end) {
        g_sampler = Sampler();
        g_sampler.fixed = false;
        g_sampler.key[0] = (uint32_t)seed;
        g_sampler.key[1] = (uint32_t)(seed >> 32);
        for (int64_t r = b; r < end; ++r) {
            const int j = height - 1 - (int)r;
            for (int i = 0; i < width; ++i) {
                Vec3 acc;
                g_sampler.pixel = (uint32_t)(r * width + i);
                for (int sidx = spp_begin; sidx < spp_begin + spp_count; ++sidx) {
                    g_sampler.sample = (uint32_t)sidx;
                    g_sampler.bounce = 0;
                    uint32_t w[4];
                    g_sampler.block(P_CAMERA, 0, w);
                    Ray ray = camera.ray(((double)i + u01(w[0])) / (double)width, ((double)j + u01(w[1])) / (double)height);
                    acc = acc + color_env(s, e, ray, max_depth, max_depth);
                }
                double* px = rgb_sum + 3 * ((size_t)r * width + i);
                px[0] += acc.x; px[1] += acc.y; px[2] += acc.z;
            }
        }
        total_rays += g_sampler.rays;
    });
    return total_rays.load();
}

// orc_first_vertex (oracle_first_vertex.cpp) with the scene's map: a miss adds its value clamped to [0, 1].
extern "C" void orc_first_vertex_env(const orc_scene* s, int width, int height, int spp_begin, int spp_count, uint64_t seed,
                                     double* albedo_sum, double* normal_sum, double* depth_sum, int n_threads) {
    Camera camera(s->camera);
    const OrcEnv* e = env_of(s);
    std::vector<const Material*> phases;
    collect_phases(s->world.get(), phases);
    run_parallel(n_threads, height, 1, [&](int64_t b, int64_t end) {
        g_sampler = Sampler();
        g_sampler.fixed = false;
        g_sampler.key[0] = (uint32_t)seed;
        g_sampler.key[1] = (uint32_t)(seed >> 32);
        for (int64_t r = b; r < end; ++r) {
            const int j = height - 1 - (int)r;
            for (int i = 0; i < width; ++i) {
                const size_t px = (size_t)r * width + i;
                g_sampler.pixel = (uint32_t)px;
                Vec3 al, nn;
                double dist = 0.0, hits = 0.0;
                for (int sidx = spp_begin; sidx < spp_begin + spp_count; ++sidx) {
                    g_sampler.sample = (uint32_t)sidx;
                    g_sampler.bounce = 0;
                    uint32_t w[4];
                    g_sampler.block(P_CAMERA, 0, w);
                    Ray ray = camera.ray(((double)i + u01(w[0])) / (double)width, ((double)j + u01(w[1])) / (double)height);
                    HitRecord rec;
                    if (s->world->hit(ray, 0.001, DBL_MAX, rec)) {
                        const Material* m = rec.material;
                        const Vec3 emitted = m->emitted(rec.u, rec.v, rec.p);
                        Vec3 att;
                        Ray scattered;
                        m->scatter(ray, rec, att, scattered);
                        if (dynamic_cast<const DiffuseLight*>(m)) att = clamp01(emitted);
                        const bool medium = std::find(phases.begin(), phases.end(), m) != phases.end();
                        al = al + att;
                        if (!medium) nn = nn + rec.normal;
                        dist += rec.t * ray.b.magnitude();
                        hits += 1.0;
                    } else {
                        al = al + clamp01(miss_value(s, e, ray));
                    }
                }
                if (albedo_sum) { double* p = albedo_sum + 3 * px; p[0] += al.x; p[1] += al.y; p[2] += al.z; }
                if (normal_sum) { double* p = normal_sum + 3 * px; p[0] += nn.x; p[1] += nn.y; p[2] += nn.z; }
                if (depth_sum) { double* p = depth_sum + 2 * px; p[0] += dist; p[1] += hits; }
            }
        }
    });
}
