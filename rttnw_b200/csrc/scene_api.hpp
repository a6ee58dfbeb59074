// scene_api.hpp — C++ host mirror of the reference's scene API (src/math/mod.rs:10-19).
//
// The reference builds a tree of trait objects (Box/Arc<dyn Hittable|Material|Texture>);
// this header offers the same constructors by the same names, but every object is a small
// handle into a SceneBuilder that records plain rtx_node / rtx_material / rtx_texture
// entries — the description rtx_scene_create() consumes. Sharing a handle is the
// reference's Arc::clone: the entry is emitted once.
//
// Rust toolchains are absent from this image; INTEGRATION.md shows the Rust binding that
// walks the real trait objects into the same description.
#pragma once
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

#include "../../include/rttnw_b200.h"

namespace rttnw {

struct Vec3f {  // src/math/vec3.rs (only what scene construction needs)
    double x = 0, y = 0, z = 0;
    Vec3f() {}
    Vec3f(double a, double b, double c) : x(a), y(b), z(c) {}
    static Vec3f repeat(double v) { return Vec3f(v, v, v); }
    Vec3f operator+(const Vec3f& r) const { return Vec3f(x + r.x, y + r.y, z + r.z); }
    Vec3f operator-(const Vec3f& r) const { return Vec3f(x - r.x, y - r.y, z - r.z); }
    double magnitude() const;
};

// SplitMix64 stands in for rand::thread_rng() at scene-construction time (SURVEY §8d).
struct SceneRng {
    uint64_t s;
    explicit SceneRng(uint64_t seed) : s(seed) {}
    uint64_t next();
    double gen();                       // rng.gen::<f64>()
    double range(double a, double b);   // rng.gen_range(a..b)
    uint32_t below(uint32_t n);
};

class SceneBuilder;
SceneBuilder& current_builder();

struct Texture { int id = -1; };
struct Material { int id = -1; };
struct Hittable {
    int id = -1;
    Hittable translate(const Vec3f& offset) const;  // Hittable::translate, hittable.rs:51-59
    Hittable rotate_y(double angle) const;          // Hittable::rotate_y, hittable.rs:60-65
};
struct Range { double start, end; };

// ---- textures (src/math/texture.rs) ----
Texture solid(const Vec3f& color);                 // impl Texture for Vec3f<Color>
struct CheckerTexture { static Texture make(Texture odd, Texture even); };
struct NoiseTexture {
    static Texture scaled(double scale, SceneRng& rng);  // NoiseTexture::scaled + Perlin::new
};
struct ImageTexture { static Texture new_(const char* path); };  // ImageTexture::new

// ---- materials (src/math/material.rs) ----
struct Lambertian {
    static Material arc(Texture albedo);
    static Material arc(const Vec3f& albedo) { return arc(solid(albedo)); }
    static Material boxed(const Vec3f& albedo) { return arc(solid(albedo)); }
};
struct Metal { static Material arc(const Vec3f& albedo, double fuzz); };
struct Dielectric { static Material arc(double refraction_index); };
struct DiffuseLight {
    static Material arc(Texture emit);
    static Material arc(const Vec3f& emit) { return arc(solid(emit)); }
};

// ---- hittables (src/math/hittable.rs) ----
Hittable Sphere(const Vec3f& center, double radius, Material material);
Hittable MovingSphere(const Vec3f& center0, const Vec3f& center1, Range time, double radius, Material material);
struct XY { static Hittable rectangle(Material m, Range p0, Range p1, double k); };
struct XZ { static Hittable rectangle(Material m, Range p0, Range p1, double k); };
struct YZ { static Hittable rectangle(Material m, Range p0, Range p1, double k); };
using Xy = XY; using Xz = XZ; using Yz = YZ;  // both spellings occur in the reference (SURVEY Q28)
struct Cube { static Hittable new_(const Vec3f& box_min, const Vec3f& box_max, Material material); };
struct List {
    std::vector<int> items;
    void push(Hittable h) { items.push_back(h.id); }
    Hittable into_hittable() const;  // emits a LIST node
};
struct BvhTree { static Hittable from(const List& list); };
struct ConstantMedium { static Hittable new_(Hittable boundary, double density, Texture phase); };

struct CameraDescriptor {  // src/math/camera.rs:5-15
    Vec3f lookfrom, lookat, view_up{0, 1, 0};
    double vertical_fov = 40, aspect_ratio = 1, aperture = 0, focus_distance = 10, open_time = 0, close_time = 1;
};

// Owns the arrays an rtx_scene_desc points into.
class SceneBuilder {
   public:
    std::vector<rtx_node> nodes;
    std::vector<int32_t> children;
    std::vector<rtx_material> materials;
    std::vector<rtx_texture> textures;
    std::vector<rtx_perlin> perlins;
    std::vector<rtx_image> images;
    std::vector<std::vector<uint8_t>> image_pixels;
    rtx_scene_desc desc{};

    struct Scope {  // makes `b` the builder the free constructors above write into
        SceneBuilder* prev;
        explicit Scope(SceneBuilder& b);
        ~Scope();
    };
    int add_node(const rtx_node& n) { nodes.push_back(n); return (int)nodes.size() - 1; }
    // Fills `desc` (pointers stay valid until the builder is modified or destroyed).
    const rtx_scene_desc& finish(Hittable world, const CameraDescriptor& cam, const Vec3f& background);
};

// ---- scenes.rs + the scene table of main.rs ----
struct SceneDefaults { int width, height, samples, max_depth; const char* name; };
bool builtin_scene_defaults(int scene_number, SceneDefaults& out);  // main.rs:66-183,255
// Builds scene 1..9 into `b`; returns false for an unknown number (main.rs:179-182).
bool builtin_scene(int scene_number, uint64_t seed, const char* earth_png_path, SceneBuilder& b);

// PNG (zlib): returns false on failure.
bool png_read_rgba8(const char* path, int& width, int& height, std::vector<uint8_t>& rgba, std::string& err);
bool png_write_rgba8(const char* path, int width, int height, const uint8_t* rgba, std::string& err);
// PFM, 1 or 3 little-endian float channels (rtx_pfm_write)
bool pfm_write(const char* path, int width, int height, int channels, const float* data, std::string& err);

}  // namespace rttnw
