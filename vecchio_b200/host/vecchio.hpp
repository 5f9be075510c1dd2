// vecchio.hpp -- host-side front end of the B200 path: the reference's scene / Hittable /
// Material / Texture API (same names, same constructor arguments), with ONE added method per
// trait: lower(), which flattens the object to the POD arrays of include/vecchio_gpu.h.
//
// The reference host is Rust; this image has no rustc, so the host side above the C ABI is
// written in C++ (rust/gpu.rs holds the equivalent, uncompiled, Rust shim).  What lives here is
// only what the reference keeps on the host: constructors, bounding_box (input of the BVH
// build), BVHNode::new (src/accel.rs:98-136), Camera::new (src/main.rs:71-109), PNG decode
// and Perlin table generation.  There is deliberately NO CPU `hit`/`scatter` here: that work
// is the GPU's (libvecchio_gpu.so); the CPU restatement used by the tests lives in oracle/.
#pragma once
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/vecchio_gpu.h"

namespace vecchio {

template <class T> using Arc = std::shared_ptr<T>;

struct LowerError : std::runtime_error {
    using std::runtime_error::runtime_error;
};

// ---------------------------------------------------------------------------------------------
// Host RNG.  The reference draws scene randomness from the unseeded rand::thread_rng()
// (src/scene.rs:183,735; src/accel.rs:99; src/material.rs:358); only the distributions can be
// kept.  gen_f32: 24-bit [0,1); gen_range: the 23-bit [1,2) construction of rand 0.7.3.
// ---------------------------------------------------------------------------------------------
class HostRng {
  public:
    explicit HostRng(uint64_t seed = 1) { reseed(seed); }
    void reseed(uint64_t seed) {
        s_ = seed * 0x9E3779B97F4A7C15ull + 0xD1B54A32D192ED03ull;
        for (int i = 0; i < 4; ++i) next_u64();
    }
    uint64_t next_u64() { // splitmix64
        uint64_t z = (s_ += 0x9E3779B97F4A7C15ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    }
    uint32_t next_u32() { return (uint32_t)(next_u64() >> 32); }
    float gen_f32() { return (float)(next_u32() >> 8) * (1.0f / 16777216.0f); }
    float gen_range(float low, float high) {
        const float scale = high - low, offset = low - scale;
        for (;;) {
            uint32_t bits = 0x3F800000u | (next_u32() >> 9);
            float v12;
            std::memcpy(&v12, &bits, 4);
            float res = v12 * scale + offset;
            if (res < high) return res;
        }
    }
    uint32_t gen_range_u32(uint32_t low, uint32_t high) { // [low, high)
        return low + (uint32_t)(((uint64_t)next_u32() * (uint64_t)(high - low)) >> 32);
    }
    template <class T> void shuffle(T* a, size_t n) { // Fisher-Yates (SliceRandom::shuffle)
        for (size_t i = n; i > 1; --i) std::swap(a[i - 1], a[gen_range_u32(0, (uint32_t)i)]);
    }

  private:
    uint64_t s_;
};
HostRng& thread_rng();         // the process-wide stand-in for rand::thread_rng()
void seed_thread_rng(uint64_t seed);

// ---------------------------------------------------------------------------------------------
// Vec3 (src/vec3.rs)
// ---------------------------------------------------------------------------------------------
struct Vec3 {
    float x = 0, y = 0, z = 0;
    Vec3() = default;
    Vec3(float x_, float y_, float z_) : x(x_), y(y_), z(z_) {}
    static Vec3 new_const(float v) { return Vec3(v, v, v); }
    static Vec3 zero() { return new_const(0.0f); }
    float dot(Vec3 v) const { return x * v.x + y * v.y + z * v.z; }
    Vec3 cross(Vec3 v) const { return Vec3(y * v.z - z * v.y, z * v.x - x * v.z, x * v.y - y * v.x); }
    float length2() const { return x * x + y * y + z * z; }
    float length() const { return std::sqrt(length2()); }
    Vec3 unit_vector() const {
        float n = std::sqrt(length2());
        return Vec3(x / n, y / n, z / n);
    }
    static Vec3 random() {
        auto& r = thread_rng();
        float a = r.gen_f32(), b = r.gen_f32(), c = r.gen_f32();
        return Vec3(a, b, c);
    }
    static Vec3 random_range(float lo, float hi) {
        auto& r = thread_rng();
        float a = r.gen_range(lo, hi), b = r.gen_range(lo, hi), c = r.gen_range(lo, hi);
        return Vec3(a, b, c);
    }
    float operator[](size_t i) const { return i == 0 ? x : (i == 1 ? y : z); }
    float& operator[](size_t i) { return i == 0 ? x : (i == 1 ? y : z); }
};
inline Vec3 operator+(Vec3 a, Vec3 b) { return Vec3(a.x + b.x, a.y + b.y, a.z + b.z); }
inline Vec3 operator-(Vec3 a, Vec3 b) { return Vec3(a.x - b.x, a.y - b.y, a.z - b.z); }
inline Vec3 operator*(Vec3 a, Vec3 b) { return Vec3(a.x * b.x, a.y * b.y, a.z * b.z); }
inline Vec3 operator*(Vec3 a, float s) { return Vec3(a.x * s, a.y * s, a.z * s); }
inline Vec3 operator/(Vec3 a, float s) { return Vec3(a.x / s, a.y / s, a.z / s); }
inline Vec3 operator-(Vec3 a) { return Vec3(-a.x, -a.y, -a.z); }

inline float to_radians(float deg) { return deg * (3.14159265358979323846f / 180.0f); }

// ---------------------------------------------------------------------------------------------
// Camera (src/main.rs:56-109).  get_ray (:111-120) runs on the GPU.
// ---------------------------------------------------------------------------------------------
struct Camera {
    Vec3 origin, lower_left_corner, horizontal, vertical, u, v, w;
    float lens_radius = 0, time0 = 0, time1 = 1;
    static Camera make(Vec3 lookfrom, Vec3 lookat, Vec3 vup, float vfov, float aspect_ratio,
                       float aperture, float focus_dist, float time0, float time1);
    vk_camera lower() const;
};

// ---------------------------------------------------------------------------------------------
// AxisBB (src/accel.rs:9-50); AxisBB::hit runs on the GPU.
// ---------------------------------------------------------------------------------------------
struct AxisBB {
    Vec3 min, max;
    AxisBB() = default;
    AxisBB(Vec3 a, Vec3 b) : min(a), max(b) {}
    static AxisBB surrounding_box(AxisBB b1, AxisBB b2);
};

class Lowering;

// ---------------------------------------------------------------------------------------------
// Texture (src/material.rs:228-434)
// ---------------------------------------------------------------------------------------------
struct Texture {
    virtual ~Texture() = default;
    virtual uint32_t lower(Lowering&) const { throw LowerError("Texture: unsupported type"); }
};
using TextureSS = Texture;

struct SolidColor : Texture {
    Vec3 color_value;
    explicit SolidColor(Vec3 c) : color_value(c) {}
    uint32_t lower(Lowering&) const override;
};
struct Checker : Texture {
    Arc<TextureSS> odd, even;
    Checker(Arc<TextureSS> o, Arc<TextureSS> e) : odd(std::move(o)), even(std::move(e)) {}
    uint32_t lower(Lowering&) const override;
};
struct ImageTexture : Texture {
    std::vector<uint8_t> buf;
    size_t width = 0, height = 0;
    explicit ImageTexture(const std::string& path); // PNG decode, src/material.rs:269-279
    uint32_t lower(Lowering&) const override;
};
struct Perlin {
    static constexpr size_t NUM_POINTS = 256;
    std::array<Vec3, NUM_POINTS> random_data;
    std::array<size_t, NUM_POINTS> perm_x, perm_y, perm_z;
    Perlin(); // src/material.rs:357-377
};
struct NoiseTexture : Texture {
    Perlin noise;
    float scale;
    explicit NoiseTexture(float s) : scale(s) {}
    uint32_t lower(Lowering&) const override;
};

// ---------------------------------------------------------------------------------------------
// Material (src/material.rs:20-226, 436-488)
// ---------------------------------------------------------------------------------------------
struct Material {
    virtual ~Material() = default;
    virtual uint32_t lower(Lowering&) const { throw LowerError("Material: unsupported type"); }
};
using MaterialSS = Material;

struct Lambertian : Material {
    Arc<TextureSS> albedo;
    explicit Lambertian(Arc<TextureSS> a) : albedo(std::move(a)) {}
    uint32_t lower(Lowering&) const override;
};
struct Metal : Material {
    Arc<TextureSS> albedo;
    float fuzz;
    Metal(Arc<TextureSS> a, float f) : albedo(std::move(a)), fuzz(f) {}
    uint32_t lower(Lowering&) const override;
};
struct Dielectric : Material {
    float ref_idx;
    explicit Dielectric(float r) : ref_idx(r) {}
    uint32_t lower(Lowering&) const override;
};
struct DiffuseLight : Material {
    Arc<TextureSS> emit;
    explicit DiffuseLight(Arc<TextureSS> e) : emit(std::move(e)) {}
    uint32_t lower(Lowering&) const override;
};
struct Isotropic : Material {
    Arc<TextureSS> albedo;
    explicit Isotropic(Arc<TextureSS> a) : albedo(std::move(a)) {}
    uint32_t lower(Lowering&) const override;
};
struct SpecDiffuse : Material {
    Arc<MaterialSS> specular, diffuse;
    float pct;
    SpecDiffuse(Arc<MaterialSS> s, Arc<MaterialSS> d, float p)
        : specular(std::move(s)), diffuse(std::move(d)), pct(p) {}
    uint32_t lower(Lowering&) const override;
};

// ---------------------------------------------------------------------------------------------
// Hittable (src/hittable.rs:33-44).  hit / pdf_value / random run on the GPU.
// ---------------------------------------------------------------------------------------------
struct Hittable {
    virtual ~Hittable() = default;
    virtual std::optional<AxisBB> bounding_box(float t0, float t1) const = 0;
    virtual vk_ref lower(Lowering&) const { throw LowerError("Hittable: unsupported type"); }
};
using HittableSS = Hittable;

struct Sphere : Hittable {
    Vec3 center;
    float radius;
    Arc<MaterialSS> material;
    Sphere(Vec3 c, float r, Arc<MaterialSS> m) : center(c), radius(r), material(std::move(m)) {}
    std::optional<AxisBB> bounding_box(float, float) const override;
    vk_ref lower(Lowering&) const override;
};
struct MovingSphere : Hittable {
    Vec3 center0, center1;
    float time0, time1, radius;
    Arc<MaterialSS> material;
    MovingSphere(Vec3 c0, Vec3 c1, float t0, float t1, float r, Arc<MaterialSS> m)
        : center0(c0), center1(c1), time0(t0), time1(t1), radius(r), material(std::move(m)) {}
    Vec3 center(float time) const;
    std::optional<AxisBB> bounding_box(float, float) const override;
    vk_ref lower(Lowering&) const override;
};
struct Rect : Hittable {
    float c0, c1, d0, d1, k;
    size_t axis0, axis1, axis2;
    Arc<MaterialSS> mat;
    Rect(float c0_, float c1_, float d0_, float d1_, float k_, size_t a0, size_t a1, size_t a2,
         Arc<MaterialSS> m)
        : c0(c0_), c1(c1_), d0(d0_), d1(d1_), k(k_), axis0(a0), axis1(a1), axis2(a2), mat(std::move(m)) {}
    static Rect XYRect(float x0, float x1, float y0, float y1, float k, Arc<MaterialSS> m) {
        return Rect(x0, x1, y0, y1, k, 0, 1, 2, std::move(m));
    }
    static Rect XZRect(float x0, float x1, float z0, float z1, float k, Arc<MaterialSS> m) {
        return Rect(x0, x1, z0, z1, k, 0, 2, 1, std::move(m));
    }
    static Rect YZRect(float y0, float y1, float z0, float z1, float k, Arc<MaterialSS> m) {
        return Rect(y0, y1, z0, z1, k, 1, 2, 0, std::move(m));
    }
    std::optional<AxisBB> bounding_box(float, float) const override;
    vk_ref lower(Lowering&) const override;
    vk_ref lower_flipped(Lowering&, bool flip) const;
};
struct FlipFace : Hittable {
    Arc<HittableSS> ptr;
    explicit FlipFace(Arc<HittableSS> p) : ptr(std::move(p)) {}
    std::optional<AxisBB> bounding_box(float t0, float t1) const override { return ptr->bounding_box(t0, t1); }
    vk_ref lower(Lowering&) const override;
};
struct Boxy : Hittable {
    Vec3 box_min, box_max;
    Arc<MaterialSS> mat; // the six sides of src/hittable.rs:325-353 are implied by (min,max,mat)
    Boxy(Vec3 p0, Vec3 p1, Arc<MaterialSS> m);
    std::optional<AxisBB> bounding_box(float, float) const override { return AxisBB(box_min, box_max); }
    vk_ref lower(Lowering&) const override;
};
struct ConstantMedium : Hittable {
    Arc<HittableSS> boundary;
    Arc<MaterialSS> phase_function;
    float neg_inv_density;
    ConstantMedium(Arc<HittableSS> b, float density, Arc<TextureSS> albedo)
        : boundary(std::move(b)), phase_function(std::make_shared<Isotropic>(std::move(albedo))),
          neg_inv_density(-1.0f / density) {}
    std::optional<AxisBB> bounding_box(float t0, float t1) const override { return boundary->bounding_box(t0, t1); }
    vk_ref lower(Lowering&) const override;
};
struct Translate : Hittable {
    Arc<HittableSS> ptr;
    Vec3 offset;
    Translate(Arc<HittableSS> p, Vec3 o) : ptr(std::move(p)), offset(o) {}
    std::optional<AxisBB> bounding_box(float t0, float t1) const override;
    vk_ref lower(Lowering&) const override;
};
struct RotateAxis : Hittable { // shared body of RotateX / RotateY / RotateZ
    Arc<HittableSS> ptr;
    float sin_theta, cos_theta;
    std::optional<AxisBB> bb;
    uint32_t kind;
    RotateAxis(Arc<HittableSS> p, float angle_deg, uint32_t kind);
    std::optional<AxisBB> bounding_box(float, float) const override { return bb; }
    vk_ref lower(Lowering&) const override;
};
struct RotateX : RotateAxis { RotateX(Arc<HittableSS> p, float a) : RotateAxis(std::move(p), a, VK_X_ROTATE_X) {} };
struct RotateY : RotateAxis { RotateY(Arc<HittableSS> p, float a) : RotateAxis(std::move(p), a, VK_X_ROTATE_Y) {} };
struct RotateZ : RotateAxis { RotateZ(Arc<HittableSS> p, float a) : RotateAxis(std::move(p), a, VK_X_ROTATE_Z) {} };

// BVHNode (src/accel.rs:52-137): built here exactly like the reference (random axis, median
// split, single-object leaves with left == right), traversed on the GPU.
struct BVHNode : Hittable {
    Arc<HittableSS> left, right;
    AxisBB bb;
    BVHNode() = default;
    static Arc<BVHNode> make(std::vector<Arc<HittableSS>>& objects) { return make(objects.data(), objects.size()); }
    static Arc<BVHNode> make(Arc<HittableSS>* objects, size_t n);
    std::optional<AxisBB> bounding_box(float, float) const override { return bb; }
    vk_ref lower(Lowering&) const override;
};

// ---------------------------------------------------------------------------------------------
// Lowering: accumulates the flat arrays of vk_scene_desc.  Shared Arcs are lowered once.
// ---------------------------------------------------------------------------------------------
class Lowering {
  public:
    std::vector<vk_node> nodes;
    std::vector<vk_sphere> spheres;
    std::vector<uint32_t> sphere_mat;
    std::vector<vk_msphere> mspheres;
    std::vector<vk_rect> rects;
    std::vector<vk_box> boxes;
    std::vector<vk_xform> xforms;
    std::vector<vk_medium> media;
    std::vector<vk_ref> lights;
    std::vector<vk_material> materials;
    std::vector<vk_texture> textures;
    std::vector<uint8_t> texels;
    std::vector<vk_perlin> perlins;
    vk_ref root = VK_REF_NONE;

    vk_ref hittable(const Arc<HittableSS>& h);
    uint32_t material(const Arc<MaterialSS>& m);
    uint32_t texture(const Arc<TextureSS>& t);
    vk_scene_desc desc() const;

    std::unordered_map<const void*, vk_ref> memo_h;      // object -> ref
    std::unordered_map<const void*, vk_ref> memo_h_flip; // Rect lowered with the flip bit
    std::unordered_map<const void*, uint32_t> memo_m, memo_t;
};

// ---------------------------------------------------------------------------------------------
// Scenes (src/scene.rs)
// ---------------------------------------------------------------------------------------------
struct CameraIter {
    virtual ~CameraIter() = default;
    virtual std::optional<Camera> next() = 0;
};
struct SceneConfig {
    std::vector<Arc<HittableSS>> world;
    std::vector<Arc<HittableSS>> lights;
    std::unique_ptr<CameraIter> cam_iter;
    float aspect_ratio = 1.0f;
};

extern std::string g_assets_dir; // where "assets/earthmap.png" etc. are looked up

SceneConfig balls_demo();
SceneConfig random_spheres_demo();
SceneConfig perlin_demo();
SceneConfig bowser_demo();
SceneConfig cornell_box();
SceneConfig final_scene();
// Authored with the same API for BASELINE.json configs 3 and 5 (not in src/scene.rs).
SceneConfig cornell_smoke();
SceneConfig stress_spheres(uint32_t grid_side);
SceneConfig api_surface_demo();     // SpecDiffuse + sphere and box lights (API surface no shipped scene uses)
SceneConfig furnace_demo(uint32_t kind); // one object (0 Lambertian, 1 Metal, 2 Dielectric, 3 white medium, 4 Lambertian in a 1000x brighter shell) inside an emitting shell: closed-form radiance
SceneConfig book1_cover();          // the book-1 final scene as sample/inoneweekend.png shows it (grey ground, brown sphere, fixed camera; legacy integrator)
SceneConfig random_spheres_cover(); // random_spheres_demo without its light: the sky-lit book-1 cover (legacy integrator)

// A scene lowered for the GPU: the boundary object of src/main.rs:168-169.
struct LoweredScene {
    Lowering low;
    std::unique_ptr<CameraIter> cam_iter;
    float aspect_ratio = 1.0f;
};
std::unique_ptr<LoweredScene> lower_scene(SceneConfig&& cfg);

} // namespace vecchio
