// oracle.cpp -- CPU restatement of vecchio's path-tracing sample loop.
//
// TEST INFRASTRUCTURE (see oracle.h).  Every function cites the reference file:line it follows
// (paths relative to the reference root).  It deliberately keeps the reference's shape --
// shared_ptr for Arc, virtual dispatch for dyn Trait, recursion in ray_color and BVHNode::hit,
// a heap-allocated PDF per bounce -- and every quirk of SURVEY.md Appendix A.  Two additions
// only: a primitive id in HitRec (the reference has none) and an explicit RNG object instead
// of rand::thread_rng() so tests can inject variates.
//
// Build: g++ -O3 -std=c++17 -fopenmp -ffp-contract=off  (Rust never contracts a*b+c).
#include "oracle.h"

#include <omp.h>

#include <chrono>
#include <cmath>
#include <cstring>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

namespace orc {

template <class T> using Arc = std::shared_ptr<T>;
static const float PI = 3.14159265358979323846f; // std::f32::consts::PI
static const float INF = INFINITY;

// ------------------------------------------------------------------------------------------
// RNG.  rand 0.7.3: gen::<f32>() is 24-bit in [0,1); gen_range(a,b) is the 23-bit [1,2)
// construction; thread_rng() is replaced by a thread-local pointer to one of these.
// ------------------------------------------------------------------------------------------
struct Rng {
    uint64_t s = 0x853c49e6748fea9bull;
    void seed(uint64_t a, uint64_t b, uint64_t c) {
        s = a * 0x9E3779B97F4A7C15ull ^ (b + 0x632BE59BD9B4E019ull) * 0xD1342543DE82EF95ull ^ (c << 1 | 1) * 0xDA942042E4DD58B5ull;
        next_u64();
        next_u64();
    }
    uint64_t next_u64() { // splitmix64
        uint64_t z = (s += 0x9E3779B97F4A7C15ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    }
    // tests can script the next words (orc_eval_batch feeds the variates the GPU hook was given)
    const uint32_t* script = nullptr;
    size_t script_n = 0, script_pos = 0;
    uint32_t next_u32() {
        if (script && script_pos < script_n) return script[script_pos++];
        return (uint32_t)(next_u64() >> 32);
    }
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
    size_t gen_index(size_t n) { return (size_t)(((uint64_t)next_u32() * (uint64_t)n) >> 32); }
    // free-flight variate of ConstantMedium::hit (src/hittable.rs:473); tests inject a table
    const float* medium_xi = nullptr;
    uint8_t medium_visits[VK_MEDIUM_XI_SLOTS] = {0};
    float gen_medium(uint32_t medium_index) {
        if (!medium_xi) return gen_f32();
        uint32_t base = (medium_index * 2u) % VK_MEDIUM_XI_SLOTS;
        uint32_t visit = medium_visits[base]++; // second test of a single-object BVH leaf -> slot+1
        return medium_xi[(base + visit) % VK_MEDIUM_XI_SLOTS];
    }
};
static thread_local Rng* tl_rng = nullptr;
static inline Rng& thread_rng() { return *tl_rng; }

struct Counters {
    uint64_t rays = 0, n_node = 0, n_sph_rej = 0, n_sph_acc = 0, n_msph = 0, n_rect_rej = 0, n_rect_acc = 0, n_box = 0,
             n_translate = 0, n_rotate = 0, n_medium = 0, n_texel = 0, n_perlin = 0, n_diffuse = 0, n_dielectric = 0,
             n_metal = 0, n_emit_or_miss = 0, n_light_pdf = 0, rays_live = 0;
};
static thread_local Counters tl_cnt;

// ------------------------------------------------------------------------------------------
// src/vec3.rs
// ------------------------------------------------------------------------------------------
struct Vec3 {
    float x = 0, y = 0, z = 0;
    Vec3() = default;
    Vec3(float a, float b, float c) : x(a), y(b), z(c) {}
    static Vec3 new_const(float v) { return Vec3(v, v, v); }                                    // :11-13
    float dot(Vec3 v) const { return x * v.x + y * v.y + z * v.z; }                             // :19-21
    Vec3 cross(Vec3 v) const { return Vec3(y * v.z - z * v.y, z * v.x - x * v.z, x * v.y - y * v.x); } // :23-29
    float length2() const { return x * x + y * y + z * z; }                                     // :31-33
    float length() const { return std::sqrt(length2()); }                                       // :35-37
    Vec3 unit_vector() const {                                                                  // :39-42
        float norm = std::sqrt(length2());
        return Vec3(x / norm, y / norm, z / norm);
    }
    static float clamp(float v, float mn, float mx) { return v < mn ? mn : (v > mx ? mx : v); } // :44-52
    float operator[](size_t i) const { return i == 0 ? x : (i == 1 ? y : z); }                  // :174-184
    float& operator[](size_t i) { return i == 0 ? x : (i == 1 ? y : z); }
    bool is_finite() const { return std::isfinite(x) && std::isfinite(y) && std::isfinite(z); }
    static Vec3 random_range(float mn, float mx) {                                              // :74-82
        Rng& r = thread_rng();
        float a = r.gen_range(mn, mx), b = r.gen_range(mn, mx), c = r.gen_range(mn, mx);
        return Vec3(a, b, c);
    }
};
static inline Vec3 operator+(Vec3 a, Vec3 b) { return Vec3(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline Vec3 operator-(Vec3 a, Vec3 b) { return Vec3(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline Vec3 operator*(Vec3 a, Vec3 b) { return Vec3(a.x * b.x, a.y * b.y, a.z * b.z); }
static inline Vec3 operator*(Vec3 a, float s) { return Vec3(a.x * s, a.y * s, a.z * s); }
static inline Vec3 operator/(Vec3 a, float s) { return Vec3(a.x / s, a.y / s, a.z / s); }
static inline Vec3 operator-(Vec3 a) { return Vec3(-a.x, -a.y, -a.z); }
// `as u32` saturates and maps NaN to 0 (src/vec3.rs:54-61)
static inline uint32_t f32_as_u32(float f) { return !(f > 0.0f) ? 0u : (f >= 4294967296.0f ? 0xFFFFFFFFu : (uint32_t)f); }
static inline size_t f32_as_usize(float f) { return !(f > 0.0f) ? (size_t)0 : (f >= 18446744073709551616.0f ? SIZE_MAX : (size_t)f); }
static void to_color(Vec3 c, uint32_t out[3]) {
    out[0] = f32_as_u32(256.0f * Vec3::clamp(std::sqrt(c.x), 0.0f, 0.999f));
    out[1] = f32_as_u32(256.0f * Vec3::clamp(std::sqrt(c.y), 0.0f, 0.999f));
    out[2] = f32_as_u32(256.0f * Vec3::clamp(std::sqrt(c.z), 0.0f, 0.999f));
}

// ------------------------------------------------------------------------------------------
// src/main.rs:31-54  Ray
// ------------------------------------------------------------------------------------------
struct Ray {
    Vec3 origin, direction;
    float time = 0.0f;
    Ray() = default;
    Ray(Vec3 o, Vec3 d) : origin(o), direction(d), time(0.0f) {}         // Ray::new, time 0
    Ray(Vec3 o, Vec3 d, float t) : origin(o), direction(d), time(t) {}  // new_with_time
    Vec3 at(float t) const { return origin + direction * t; }
};

// ------------------------------------------------------------------------------------------
// src/util.rs
// ------------------------------------------------------------------------------------------
static inline float fmin_(float a, float b) { return std::fmin(a, b); } // :6-8  f32::min
static inline float fmax_(float a, float b) { return std::fmax(a, b); } // :10-12 f32::max
static Vec3 reflect(Vec3 v, Vec3 n) { return v - n * v.dot(n) * 2.0f; } // :14-16
static Vec3 refract(Vec3 uv, Vec3 n, float etai_over_etat) {            // :18-23
    float cos_theta = -uv.dot(n);
    Vec3 r_out_parallel = (uv + n * cos_theta) * etai_over_etat;
    Vec3 r_out_perp = n * -std::sqrt(1.0f - r_out_parallel.length2());
    return r_out_parallel + r_out_perp;
}
static float schlick(float cosine, float ref_idx) { // :25-29
    float r0 = (1.0f - ref_idx) / (1.0f + ref_idx);
    r0 = r0 * r0;
    return r0 + (1.0f - r0) * std::pow(1.0f - cosine, 5.0f);
}
static Vec3 random_in_unit_sphere() { // :31-39
    for (;;) {
        Vec3 p = Vec3::random_range(-1.0f, 1.0f);
        if (p.length2() >= 1.0f) continue;
        return p;
    }
}
static Vec3 random_in_unit_disk() { // :41-50
    Rng& rng = thread_rng();
    for (;;) {
        float a = rng.gen_range(-1.0f, 1.0f), b = rng.gen_range(-1.0f, 1.0f);
        Vec3 p(a, b, 0.0f);
        if (p.length2() >= 1.0f) continue;
        return p;
    }
}
static Vec3 random_cosine_direction() { // :52-63
    Rng& rng = thread_rng();
    float r1 = rng.gen_f32();
    float r2 = rng.gen_f32();
    float z = std::sqrt(1.0f - r2);
    float phi = 2.0f * r1 * PI;
    float x = std::cos(phi) * std::sqrt(r2);
    float y = std::sin(phi) * std::sqrt(r2);
    return Vec3(x, y, z);
}
struct ONB { // :65-111
    Vec3 u, v, w;
    Vec3 local(Vec3 a) const { return u * a.x + v * a.y + w * a.z; }
    static ONB new_from_w(Vec3 n) {
        ONB o;
        o.w = n.unit_vector();
        Vec3 a = std::fabs(o.w.x) > 0.9f ? Vec3(0, 1, 0) : Vec3(1, 0, 0);
        o.v = o.w.cross(a).unit_vector();
        o.u = o.w.cross(o.v);
        return o;
    }
};

struct Hittable;
struct PDF { // :113-117
    virtual ~PDF() = default;
    virtual float value(Vec3 direction) const = 0;
    virtual Vec3 generate() const = 0;
};
struct CosinePDF : PDF { // :121-147
    ONB uvw;
    explicit CosinePDF(Vec3 w) : uvw(ONB::new_from_w(w)) {}
    float value(Vec3 direction) const override {
        float cos = direction.unit_vector().dot(uvw.w);
        return cos <= 0.0f ? 0.0f : cos / PI;
    }
    Vec3 generate() const override { return uvw.local(random_cosine_direction()); }
};

// ------------------------------------------------------------------------------------------
// src/hittable.rs:11-44  HitRec, Hittable
// ------------------------------------------------------------------------------------------
struct Material;
struct HitRec {
    Vec3 p, normal;
    float t = 0, u = 0, v = 0;
    bool front = false;
    Arc<Material> material;
    vk_ref prim = VK_REF_NONE; // addition: id of the leaf record (the reference has none)
    uint32_t face = 0;
    HitRec(Vec3 p_, Vec3 n_, float t_, float u_, float v_, bool f_, Arc<Material> m_)
        : p(p_), normal(n_), t(t_), u(u_), v(v_), front(f_), material(std::move(m_)) {}
    void set_face_normal(const Ray& r, Vec3 outward_normal) { // :23-30
        front = r.direction.dot(outward_normal) < 0.0f;
        normal = front ? outward_normal : -outward_normal;
    }
};
struct AxisBB;
struct Hittable { // :33-42
    virtual ~Hittable() = default;
    virtual std::optional<HitRec> hit(const Ray& r, float tmin, float tmax) const = 0;
    virtual float pdf_value(Vec3, Vec3) const { return 0.0f; }
    virtual Vec3 random(Vec3) const { return Vec3(1.0f, 0.0f, 0.0f); }
};
using HittableList = std::vector<Arc<Hittable>>;

struct HittablePDF : PDF { // src/util.rs:149-162
    Arc<Hittable> ptr;
    Vec3 o;
    HittablePDF(Arc<Hittable> p, Vec3 o_) : ptr(std::move(p)), o(o_) {}
    float value(Vec3 direction) const override { return ptr->pdf_value(o, direction); }
    Vec3 generate() const override { return ptr->random(o); }
};
struct MixturePDF : PDF { // src/util.rs:164-186
    Arc<PDF> ptr1, ptr2;
    float f1, f2;
    MixturePDF(Arc<PDF> p1, float f1_, Arc<PDF> p2, float f2_) : ptr1(std::move(p1)), ptr2(std::move(p2)), f1(f1_), f2(f2_) {}
    float value(Vec3 d) const override { return f1 * ptr1->value(d) + f2 * ptr2->value(d); }
    Vec3 generate() const override {
        Rng& rng = thread_rng();
        if (rng.gen_f32() < f1) return ptr1->generate();
        return ptr2->generate();
    }
};

// ------------------------------------------------------------------------------------------
// src/material.rs: textures :228-434
// ------------------------------------------------------------------------------------------
struct Texture {
    virtual ~Texture() = default;
    virtual Vec3 value(float u, float v, Vec3 p) const = 0;
};
struct SolidColor : Texture { // :233-242
    Vec3 color_value;
    explicit SolidColor(Vec3 c) : color_value(c) {}
    Vec3 value(float, float, Vec3) const override { return color_value; }
};
struct Checker : Texture { // :244-259
    Arc<Texture> odd, even;
    Vec3 value(float u, float v, Vec3 p) const override {
        float sins = std::sin(10.0f * p.x) * std::sin(10.0f * p.y) * std::sin(10.0f * p.z);
        return sins < 0.0f ? odd->value(u, v, p) : even->value(u, v, p);
    }
};
struct ImageTexture : Texture { // :261-304
    const uint8_t* buf = nullptr;
    size_t width = 0, height = 0;
    Vec3 value(float u, float v, Vec3) const override {
        const size_t BPP = 3;
        tl_cnt.n_texel++;
        u = Vec3::clamp(u, 0.0f, 1.0f);
        v = 1.0f - Vec3::clamp(v, 0.0f, 1.0f);
        size_t i = f32_as_usize(u * (float)width);
        size_t j = f32_as_usize(v * (float)height);
        if (i >= width) i = width - 1;
        if (j >= height) j = height - 1;
        size_t buf_start = j * width * BPP + i * BPP;
        const uint8_t* pix = buf + buf_start;
        float color_scale = 1.0f / 255.0f;
        return Vec3(color_scale * (float)pix[0], color_scale * (float)pix[1], color_scale * (float)pix[2]);
    }
};
static float perlin_interp(const Vec3 c[2][2][2], float u, float v, float w) { // :331-352
    float accum = 0.0f;
    float uu = u * u * (3.0f - 2.0f * u);
    float vv = v * v * (3.0f - 2.0f * v);
    float ww = w * w * (3.0f - 2.0f * w);
    for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 2; ++j)
            for (int k = 0; k < 2; ++k) {
                float fi = (float)i, fj = (float)j, fk = (float)k;
                Vec3 weight_v(u - fi, v - fj, w - fk);
                accum += (fi * uu + (1.0f - fi) * (1.0f - uu)) * (fj * vv + (1.0f - fj) * (1.0f - vv)) *
                         (fk * ww + (1.0f - fk) * (1.0f - ww)) * c[i][j][k].dot(weight_v);
            }
    return accum;
}
struct Perlin { // :306-311, :379-413
    Vec3 random_data[256];
    size_t perm_x[256], perm_y[256], perm_z[256];
    float noise(Vec3 p) const {
        tl_cnt.n_perlin++;
        float u = p.x - std::floor(p.x);
        float v = p.y - std::floor(p.y);
        float w = p.z - std::floor(p.z);
        Vec3 c[2][2][2];
        size_t i = f32_as_usize(std::floor(p.x)); // saturating cast: negatives -> 0 (Q16)
        size_t j = f32_as_usize(std::floor(p.y));
        size_t k = f32_as_usize(std::floor(p.z));
        for (size_t di = 0; di < 2; ++di)
            for (size_t dj = 0; dj < 2; ++dj)
                for (size_t dk = 0; dk < 2; ++dk)
                    c[di][dj][dk] = random_data[perm_x[(i + di) & 255] ^ perm_y[(j + dj) & 255] ^ perm_z[(k + dk) & 255]];
        return perlin_interp(c, u, v, w);
    }
    float turb(Vec3 p, size_t depth) const {
        float accum = 0.0f;
        Vec3 temp_p = p;
        float weight = 1.0f;
        for (size_t d = 0; d < depth; ++d) {
            accum += weight * noise(temp_p);
            weight *= 0.5f;
            temp_p = temp_p * 2.0f;
        }
        return std::fabs(accum);
    }
};
struct NoiseTexture : Texture { // :416-434
    Perlin noise;
    float scale = 1.0f;
    Vec3 value(float, float, Vec3 p) const override {
        return Vec3::new_const(1.0f) * 0.5f * (1.0f + std::sin(scale * p.z + 10.0f * noise.turb(p, 7)));
    }
};

// ------------------------------------------------------------------------------------------
// src/material.rs: materials :13-226, :436-488
// ------------------------------------------------------------------------------------------
struct ScatterRec { // :13-18
    std::optional<Ray> specular_ray;
    Vec3 attenuation;
    Arc<PDF> pdf;
};
static bool g_scatter_unwrap_panic = false; // set where the reference would panic; orc_render reports it
struct Material { // :20-41
    virtual ~Material() = default;
    // the book-1/2 method, :21-28: by default built from scatter_with_pdf (`specular_ray.unwrap()`: a
    // material whose scatter_with_pdf has no specular ray panics there -- reported as an error here)
    virtual std::optional<std::pair<Vec3, Ray>> scatter(const Ray& r, const HitRec& rec) const {
        if (auto srec = scatter_with_pdf(r, rec)) {
            if (!srec->specular_ray) { // `unwrap()` on None panics in the reference (src/material.rs:23)
                g_scatter_unwrap_panic = true;
                return std::nullopt;
            }
            return std::make_pair(srec->attenuation, *srec->specular_ray);
        }
        return std::nullopt;
    }
    virtual std::optional<ScatterRec> scatter_with_pdf(const Ray&, const HitRec&) const { return std::nullopt; }
    virtual float scattering_pdf(const Ray&, const HitRec&, const Ray&) const { return 0.0f; }
    virtual Vec3 emitted(const HitRec&, float, float, Vec3) const { return Vec3::new_const(0.0f); }
};
static float cosine_scattering_pdf(const HitRec& rec, const Ray& s) { // :100-108 == :456-464
    float cos = rec.normal.dot(s.direction.unit_vector());
    return cos < 0.0f ? 0.0f : cos / PI;
}
struct Lambertian : Material { // :45-109
    Arc<Texture> albedo;
    static Vec3 random() { // :51-58: a uniform point on the unit sphere
        Rng& rng = thread_rng();
        float a = rng.gen_range(0.0f, 2.0f * PI);
        float z = rng.gen_range(-1.0f, 1.0f);
        float r = std::sqrt(1.0f - z * z);
        return Vec3(r * std::cos(a), r * std::sin(a), z);
    }
    std::optional<std::pair<Vec3, Ray>> scatter(const Ray& r, const HitRec& rec) const override { // :85-90
        Vec3 scatter_direction = rec.normal + Lambertian::random();
        Ray scattered(rec.p, scatter_direction, r.time);
        return std::make_pair(albedo->value(rec.u, rec.v, rec.p), scattered);
    }
    std::optional<ScatterRec> scatter_with_pdf(const Ray&, const HitRec& rec) const override {
        tl_cnt.n_diffuse++;
        return ScatterRec{std::nullopt, albedo->value(rec.u, rec.v, rec.p), std::make_shared<CosinePDF>(rec.normal)};
    }
    float scattering_pdf(const Ray&, const HitRec& rec, const Ray& s) const override { return cosine_scattering_pdf(rec, s); }
};
struct Metal : Material { // :111-142
    Arc<Texture> albedo;
    float fuzz = 0.0f;
    std::optional<std::pair<Vec3, Ray>> scatter(const Ray& r, const HitRec& rec) const override { // :118-132
        Vec3 reflected = reflect(r.direction.unit_vector(), rec.normal);
        Ray scattered(rec.p, reflected + random_in_unit_sphere() * fuzz, r.time); // keeps r.time here
        Vec3 attenuation = albedo->value(rec.u, rec.v, rec.p);
        if (scattered.direction.dot(rec.normal) > 0.0f) return std::make_pair(attenuation, scattered);
        return std::nullopt;
    }
    std::optional<ScatterRec> scatter_with_pdf(const Ray& r, const HitRec& rec) const override {
        tl_cnt.n_metal++;
        Vec3 reflected = reflect(r.direction.unit_vector(), rec.normal);
        // Ray::new -> time 0 (Q6); no below-surface rejection
        Ray spec(rec.p, reflected + random_in_unit_sphere() * fuzz);
        return ScatterRec{spec, albedo->value(rec.u, rec.v, rec.p), std::make_shared<CosinePDF>(rec.normal)};
    }
};
struct Dielectric : Material { // :144-207
    float ref_idx = 1.5f;
    std::optional<ScatterRec> scatter_with_pdf(const Ray& r, const HitRec& rec) const override {
        tl_cnt.n_dielectric++;
        Rng& rng = thread_rng();
        ScatterRec srec{std::nullopt, Vec3::new_const(1.0f), std::make_shared<CosinePDF>(rec.normal)};
        float etai_over_etat = rec.front ? 1.0f / ref_idx : ref_idx;
        Vec3 unit_direction = r.direction.unit_vector();
        float cos_theta = fmin_((-unit_direction).dot(rec.normal), 1.0f);
        float sin_theta = std::sqrt(1.0f - cos_theta * cos_theta);
        if (etai_over_etat * sin_theta > 1.0f) {
            srec.specular_ray = Ray(rec.p, reflect(unit_direction, rec.normal), r.time);
            return srec;
        }
        float reflect_prob = schlick(cos_theta, etai_over_etat);
        if (rng.gen_f32() < reflect_prob) {
            srec.specular_ray = Ray(rec.p, reflect(unit_direction, rec.normal), r.time);
            return srec;
        }
        srec.specular_ray = Ray(rec.p, refract(unit_direction, rec.normal, etai_over_etat), r.time);
        return srec;
    }
};
struct DiffuseLight : Material { // :209-226
    Arc<Texture> emit;
    std::optional<std::pair<Vec3, Ray>> scatter(const Ray&, const HitRec&) const override { return std::nullopt; } // :215-217
    Vec3 emitted(const HitRec& rec, float u, float v, Vec3 p) const override {
        return rec.front ? emit->value(u, v, p) : Vec3::new_const(0.0f);
    }
};
struct Isotropic : Material { // :436-465  (a cosine lobe about rec.normal, Q8)
    Arc<Texture> albedo;
    std::optional<std::pair<Vec3, Ray>> scatter(const Ray& r, const HitRec& rec) const override { // :442-446
        Ray scattered(rec.p, random_in_unit_sphere(), r.time);
        return std::make_pair(albedo->value(rec.u, rec.v, rec.p), scattered);
    }
    std::optional<ScatterRec> scatter_with_pdf(const Ray&, const HitRec& rec) const override {
        tl_cnt.n_diffuse++;
        return ScatterRec{std::nullopt, albedo->value(rec.u, rec.v, rec.p), std::make_shared<CosinePDF>(rec.normal)};
    }
    float scattering_pdf(const Ray&, const HitRec& rec, const Ray& s) const override { return cosine_scattering_pdf(rec, s); }
};
struct SpecDiffuse : Material { // :467-488
    Arc<Material> specular, diffuse;
    float pct = 0.0f;
    std::optional<ScatterRec> scatter_with_pdf(const Ray& r, const HitRec& rec) const override {
        Rng& rng = thread_rng();
        if (rng.gen_f32() < pct) return specular->scatter_with_pdf(r, rec);
        return diffuse->scatter_with_pdf(r, rec);
    }
    float scattering_pdf(const Ray& r, const HitRec& rec, const Ray& s) const override { return diffuse->scattering_pdf(r, rec, s); }
};

// ------------------------------------------------------------------------------------------
// src/accel.rs:9-35  AxisBB
// ------------------------------------------------------------------------------------------
struct AxisBB {
    Vec3 min, max;
    bool hit(const Ray& r, float tmin, float tmax) const {
        tl_cnt.n_node++;
        float tmin_local = tmin, tmax_local = tmax;
        for (size_t a = 0; a < 3; ++a) {
            float t0 = fmin_((min[a] - r.origin[a]) / r.direction[a], (max[a] - r.origin[a]) / r.direction[a]);
            float t1 = fmax_((min[a] - r.origin[a]) / r.direction[a], (max[a] - r.origin[a]) / r.direction[a]);
            tmin_local = fmax_(t0, tmin_local);
            tmax_local = fmin_(t1, tmax_local);
            if (tmax_local <= tmin_local) return false;
        }
        return true;
    }
};

// ------------------------------------------------------------------------------------------
// src/hittable.rs
// ------------------------------------------------------------------------------------------
static void spherical(Vec3 p, float& u, float& v) { // :54-61
    float phi = std::atan2(p.z, p.x);
    float theta = std::asin(p.y);
    u = 1.0f - ((phi + PI) / (2.0f * PI));
    v = (theta + PI / 2.0f) / PI;
}
static Vec3 random_to_sphere(float radius, float distance_squared) { // :123-134 (keeps the (1-z*z) bug, Q18)
    Rng& rng = thread_rng();
    float r1 = rng.gen_f32();
    float r2 = rng.gen_f32();
    float z = 1.0f + r2 * (std::sqrt(1.0f - radius * radius / distance_squared) - 1.0f);
    float phi = 2.0f * PI * r1;
    float x = std::cos(phi) * (1.0f - z * z);
    float y = std::sin(phi) * (1.0f - z * z);
    return Vec3(x, y, z);
}
struct Sphere : Hittable { // :46-121
    Vec3 center;
    float radius = 0;
    Arc<Material> material;
    vk_ref id = VK_REF_NONE;
    std::optional<HitRec> hit(const Ray& r, float tmin, float tmax) const override {
        Vec3 oc = r.origin - center;
        float a = r.direction.length2();
        float half_b = oc.dot(r.direction);
        float c = oc.length2() - radius * radius;
        float discriminant = half_b * half_b - a * c;
        if (discriminant > 0.0f) {
            float root = std::sqrt(discriminant);
            const float temps[2] = {(-half_b - root) / a, (-half_b + root) / a};
            for (float temp : temps) {
                if (tmin < temp && temp < tmax) {
                    tl_cnt.n_sph_acc++;
                    HitRec ret(r.at(temp), (r.at(temp) - center) / radius, temp, 0.0f, 0.0f, false, material);
                    ret.set_face_normal(r, (ret.p - center) / radius);
                    spherical((ret.p - center) / radius, ret.u, ret.v);
                    ret.prim = id;
                    return ret;
                }
            }
        }
        tl_cnt.n_sph_rej++;
        return std::nullopt;
    }
    float pdf_value(Vec3 o, Vec3 d) const override { // :104-113
        if (hit(Ray(o, d), 0.001f, INF)) {
            float cos_theta_max = std::sqrt(1.0f - radius * radius / (center - o).length2());
            float solid_angle = 2.0f * PI * (1.0f - cos_theta_max);
            return 1.0f / solid_angle;
        }
        return 0.0f;
    }
    Vec3 random(Vec3 o) const override { // :115-120
        Vec3 direction = center - o;
        float distance_squared = direction.length2();
        ONB uvw = ONB::new_from_w(direction);
        return uvw.local(random_to_sphere(radius, distance_squared));
    }
};
struct MovingSphere : Hittable { // :136-197
    Vec3 center0, center1;
    float time0 = 0, time1 = 1, radius = 0;
    Arc<Material> material;
    vk_ref id = VK_REF_NONE;
    Vec3 center(float time) const { return center0 + (center1 - center0) * ((time - time0) / (time1 - time0)); } // :147-150
    std::optional<HitRec> hit(const Ray& r, float tmin, float tmax) const override {
        tl_cnt.n_msph++;
        Vec3 oc = r.origin - center(r.time);
        float a = r.direction.length2();
        float half_b = oc.dot(r.direction);
        float c = oc.length2() - radius * radius;
        float discriminant = half_b * half_b - a * c;
        if (discriminant > 0.0f) {
            float root = std::sqrt(discriminant);
            const float temps[2] = {(-half_b - root) / a, (-half_b + root) / a};
            for (float temp : temps) {
                if (tmin < temp && temp < tmax) {
                    HitRec ret(r.at(temp), (r.at(temp) - center(r.time)) / radius, temp, 0.0f, 0.0f, false, material);
                    ret.set_face_normal(r, (ret.p - center(r.time)) / radius);
                    spherical((ret.p - center(r.time)) / radius, ret.u, ret.v);
                    ret.prim = id;
                    return ret;
                }
            }
        }
        return std::nullopt;
    }
};
struct Rect : Hittable { // :199-292
    float c0 = 0, c1 = 0, d0 = 0, d1 = 0, k = 0;
    size_t axis0 = 0, axis1 = 1, axis2 = 2;
    Arc<Material> mat;
    vk_ref id = VK_REF_NONE;
    uint32_t face = 0;
    std::optional<HitRec> hit(const Ray& r, float tmin, float tmax) const override {
        float t = (k - r.origin[axis2]) / r.direction[axis2];
        if (t < tmin || t > tmax) {
            tl_cnt.n_rect_rej++;
            return std::nullopt;
        }
        float a = r.origin[axis0] + t * r.direction[axis0];
        float b = r.origin[axis1] + t * r.direction[axis1];
        if (a < c0 || a > c1 || b < d0 || b > d1) {
            tl_cnt.n_rect_rej++;
            return std::nullopt;
        }
        tl_cnt.n_rect_acc++;
        Vec3 outward_normal = Vec3::new_const(0.0f);
        outward_normal[axis2] = 1.0f;
        float u = (a - c0) / (c1 - c0);
        float v = (b - d0) / (d1 - d0);
        HitRec ret(r.at(t), Vec3::new_const(0.0f), t, u, v, false, mat);
        ret.set_face_normal(r, outward_normal);
        ret.prim = id;
        ret.face = face;
        return ret;
    }
    float pdf_value(Vec3 origin, Vec3 v) const override { // :271-282
        tl_cnt.n_light_pdf++;
        const Counters keep = tl_cnt;
        auto rec = hit(Ray(origin, v), 0.001f, INF);
        tl_cnt = keep; // this rect test is counted in n_light_pdf, not in n_rect_*
        if (rec) {
            float area = (c1 - c0) * (d1 - d0);
            float distance_squared = rec->t * rec->t * v.length2();
            float cosine = std::fabs(v.dot(rec->normal)) / v.length();
            return distance_squared / (cosine * area);
        }
        return 0.0f;
    }
    Vec3 random(Vec3 origin) const override { // :284-291
        Rng& rng = thread_rng();
        Vec3 random_point = Vec3::new_const(0.0f);
        random_point[axis0] = rng.gen_range(c0, c1);
        random_point[axis1] = rng.gen_range(d0, d1);
        random_point[axis2] = k;
        return random_point - origin;
    }
};
struct FlipFace : Hittable { // :294-312 (pdf_value / random fall back to the trait defaults)
    Arc<Hittable> ptr;
    explicit FlipFace(Arc<Hittable> p) : ptr(std::move(p)) {}
    std::optional<HitRec> hit(const Ray& r, float tmin, float tmax) const override {
        if (auto h = ptr->hit(r, tmin, tmax)) {
            h->front = !h->front;
            return h;
        }
        return std::nullopt;
    }
};
// impl Hittable for Vec<Arc<HittableSS>> :380-434
static std::optional<HitRec> list_hit(const HittableList& l, const Ray& r, float tmin, float tmax) {
    float closest_dist = tmax;
    std::optional<HitRec> closest_rec;
    for (auto& w : l) {
        if (auto rec = w->hit(r, tmin, closest_dist)) {
            if (rec->t < closest_dist) {
                closest_dist = rec->t;
                closest_rec = std::move(rec);
            }
        }
    }
    return closest_rec;
}
static float list_pdf_value(const HittableList& l, Vec3 o, Vec3 v) { // :420-427
    float weight = 1.0f / (float)l.size();
    float sum = 0.0f;
    for (auto& obj : l) sum += weight * obj->pdf_value(o, v);
    return sum;
}
static Vec3 list_random(const HittableList& l, Vec3 o) { // :429-433  (choose() panics on empty)
    Rng& rng = thread_rng();
    return l[rng.gen_index(l.size())]->random(o);
}
struct ListHittable : Hittable {
    HittableList items;
    std::optional<HitRec> hit(const Ray& r, float tmin, float tmax) const override { return list_hit(items, r, tmin, tmax); }
    float pdf_value(Vec3 o, Vec3 v) const override { return list_pdf_value(items, o, v); }
    Vec3 random(Vec3 o) const override { return list_random(items, o); }
};
struct Boxy : Hittable { // :314-378
    HittableList sides;
    Boxy(Vec3 p0, Vec3 p1, Arc<Material> mat, vk_ref id) {
        auto side = [&](Rect r, uint32_t face, bool flip) -> Arc<Hittable> {
            r.mat = mat;
            r.id = id;
            r.face = face;
            auto p = std::make_shared<Rect>(r);
            if (flip) return std::make_shared<FlipFace>(p);
            return p;
        };
        auto mk = [](float c0, float c1, float d0, float d1, float k, size_t a0, size_t a1, size_t a2) {
            Rect r;
            r.c0 = c0; r.c1 = c1; r.d0 = d0; r.d1 = d1; r.k = k;
            r.axis0 = a0; r.axis1 = a1; r.axis2 = a2;
            return r;
        };
        sides = {side(mk(p0.x, p1.x, p0.y, p1.y, p1.z, 0, 1, 2), 0, false), side(mk(p0.x, p1.x, p0.y, p1.y, p0.z, 0, 1, 2), 1, true),
                 side(mk(p0.x, p1.x, p0.z, p1.z, p1.y, 0, 2, 1), 2, false), side(mk(p0.x, p1.x, p0.z, p1.z, p0.y, 0, 2, 1), 3, true),
                 side(mk(p0.y, p1.y, p0.z, p1.z, p1.x, 1, 2, 0), 4, false), side(mk(p0.y, p1.y, p0.z, p1.z, p0.x, 1, 2, 0), 5, true)};
    }
    std::optional<HitRec> hit(const Ray& r, float tmin, float tmax) const override {
        tl_cnt.n_box++;
        return list_hit(sides, r, tmin, tmax);
    }
    float pdf_value(Vec3 o, Vec3 v) const override { return list_pdf_value(sides, o, v); }
    Vec3 random(Vec3 o) const override { return list_random(sides, o); }
};
struct ConstantMedium : Hittable { // :436-498
    Arc<Hittable> boundary;
    Arc<Material> phase_function;
    float neg_inv_density = 0;
    vk_ref id = VK_REF_NONE;
    std::optional<HitRec> hit(const Ray& r, float tmin, float tmax) const override {
        tl_cnt.n_medium++;
        Rng& rng = thread_rng();
        if (auto rec1 = boundary->hit(r, -INF, INF)) {
            if (auto rec2 = boundary->hit(r, rec1->t + 0.0001f, INF)) {
                if (rec1->t < tmin) rec1->t = tmin;
                if (rec2->t > tmax) rec2->t = tmax;
                if (rec1->t >= rec2->t) return std::nullopt;
                if (rec1->t < 0.0f) rec1->t = 0.0f;
                float ray_length = r.direction.length();
                float distance_inside_boundary = (rec2->t - rec1->t) * ray_length;
                float hit_distance = neg_inv_density * std::log(rng.gen_medium(VK_REF_INDEX(id)));
                if (hit_distance > distance_inside_boundary) return std::nullopt;
                float t = rec1->t + hit_distance / ray_length;
                HitRec out(r.at(t), Vec3(1.0f, 0.0f, 0.0f), t, rec1->u, rec1->v, true, phase_function);
                out.prim = id;
                return out;
            }
        }
        return std::nullopt;
    }
};
struct Translate : Hittable { // :500-532
    Arc<Hittable> ptr;
    Vec3 offset;
    std::optional<HitRec> hit(const Ray& r, float tmin, float tmax) const override {
        tl_cnt.n_translate++;
        Ray moved_r(r.origin - offset, r.direction, r.time);
        if (auto rec = ptr->hit(moved_r, tmin, tmax)) {
            HitRec moved_rec(rec->p + offset, rec->normal, rec->t, rec->u, rec->v, rec->front, rec->material);
            moved_rec.prim = rec->prim;
            moved_rec.face = rec->face;
            moved_rec.set_face_normal(moved_r, rec->normal);
            return moved_rec;
        }
        return std::nullopt;
    }
};
struct Rotate : Hittable { // RotateY :578-624, RotateX :675-713, RotateZ :764-802
    Arc<Hittable> ptr;
    float sin_theta = 0, cos_theta = 1;
    uint32_t kind = VK_X_ROTATE_Y;
    // world -> object and object -> world, per axis (Q10)
    void fwd(Vec3& q) const {
        Vec3 s = q;
        if (kind == VK_X_ROTATE_Y) {
            q.x = cos_theta * s.x - sin_theta * s.z;
            q.z = sin_theta * s.x + cos_theta * s.z;
        } else if (kind == VK_X_ROTATE_X) {
            q.y = cos_theta * s.y + sin_theta * s.z;
            q.z = -sin_theta * s.y + cos_theta * s.z;
        } else {
            q.x = cos_theta * s.x + sin_theta * s.y;
            q.y = -sin_theta * s.x + cos_theta * s.y;
        }
    }
    void back(Vec3& q) const {
        Vec3 s = q;
        if (kind == VK_X_ROTATE_Y) {
            q.x = cos_theta * s.x + sin_theta * s.z;
            q.z = -sin_theta * s.x + cos_theta * s.z;
        } else if (kind == VK_X_ROTATE_X) {
            q.y = cos_theta * s.y - sin_theta * s.z;
            q.z = sin_theta * s.y + cos_theta * s.z;
        } else {
            q.x = cos_theta * s.x - sin_theta * s.y;
            q.y = sin_theta * s.x + cos_theta * s.y;
        }
    }
    std::optional<HitRec> hit(const Ray& r, float tmin, float tmax) const override {
        tl_cnt.n_rotate++;
        Vec3 origin = r.origin, direction = r.direction;
        fwd(origin);
        fwd(direction);
        Ray rotated_r(origin, direction, r.time);
        if (auto rec = ptr->hit(rotated_r, tmin, tmax)) {
            Vec3 p = rec->p, normal = rec->normal;
            back(p);
            back(normal);
            HitRec out_rec(p, normal, rec->t, rec->u, rec->v, rec->front, rec->material);
            out_rec.prim = rec->prim;
            out_rec.face = rec->face;
            out_rec.set_face_normal(rotated_r, normal); // object-space ray vs world-space normal (Q9)
            return out_rec;
        }
        return std::nullopt;
    }
};

// ------------------------------------------------------------------------------------------
// src/accel.rs:52-83  BVHNode::hit
// ------------------------------------------------------------------------------------------
struct BVHNode : Hittable {
    Arc<Hittable> left, right;
    AxisBB bb;
    std::optional<HitRec> hit(const Ray& r, float tmin, float tmax) const override {
        if (!bb.hit(r, tmin, tmax)) return std::nullopt;
        auto rec_left = left->hit(r, tmin, tmax);
        float tmax_new = rec_left ? rec_left->t : tmax;
        auto rec_right = right->hit(r, tmin, tmax_new);
        if (rec_left && rec_right) return rec_left->t < rec_right->t ? rec_left : rec_right; // tie -> right
        if (rec_left) return rec_left;
        if (rec_right) return rec_right;
        return std::nullopt;
    }
};

// ------------------------------------------------------------------------------------------
// src/main.rs:56-153  Camera::get_ray, ray_color
// ------------------------------------------------------------------------------------------
struct Camera {
    Vec3 origin, lower_left_corner, horizontal, vertical, u, v, w;
    float lens_radius = 0, time0 = 0, time1 = 1;
    Ray get_ray(float s, float t) const { // :111-120
        Rng& rng = thread_rng();
        Vec3 rd = random_in_unit_disk() * lens_radius;
        Vec3 offset = u * rd.x + v * rd.y;
        Vec3 o = origin + offset;
        Vec3 d = lower_left_corner + horizontal * s + vertical * t - origin - offset;
        return Ray(o, d, rng.gen_range(time0, time1));
    }
};

struct RayTap { // optional recorder of every traced segment (orc_harvest_rays)
    vk_ray* out = nullptr;
    size_t cap = 0, n = 0;
};
static thread_local RayTap* tl_tap = nullptr;

static Vec3 sky_color(const Ray& r);

// `live` is instrumentation only: false once the path's accumulated weight is exactly zero or
// non-finite, i.e. for segments the reference still traces although they cannot change the pixel.
// `sky`: a miss returns the book-1 sky of the ray that missed (as ray_color_legacy and the GPU's miss_color do), not
// the constant background.
static Vec3 ray_color(const Ray& r, const Arc<Hittable>& world, const Arc<Hittable>& lights, uint32_t depth,
                      uint32_t max_depth, Vec3 background, bool sky, bool live = true) { // :123-153
    if (depth > max_depth) return Vec3::new_const(0.0f);
    tl_cnt.rays++;
    if (live) tl_cnt.rays_live++;
    if (tl_tap && tl_tap->n < tl_tap->cap) {
        vk_ray& o = tl_tap->out[tl_tap->n++];
        o.origin[0] = r.origin.x; o.origin[1] = r.origin.y; o.origin[2] = r.origin.z;
        o.direction[0] = r.direction.x; o.direction[1] = r.direction.y; o.direction[2] = r.direction.z;
        o.time = r.time; o.tmin = 0.001f; o.tmax = INF;
    }
    if (auto c = world->hit(r, 0.001f, INF)) {
        Vec3 emitted = c->material->emitted(*c, c->u, c->v, c->p);
        if (auto srec = c->material->scatter_with_pdf(r, *c)) {
            if (srec->specular_ray) // Specular!  (emitted is dropped, Q2)
                return srec->attenuation * ray_color(*srec->specular_ray, world, lights, depth + 1, max_depth, background, sky,
                                                     live && !(srec->attenuation.x == 0.0f && srec->attenuation.y == 0.0f && srec->attenuation.z == 0.0f));
            auto p_important = std::make_shared<HittablePDF>(lights, c->p);
            MixturePDF p(p_important, 0.5f, srec->pdf, 0.5f);
            Ray scattered(c->p, p.generate(), r.time);
            float pdf = p.value(scattered.direction);
            Vec3 w = srec->attenuation * c->material->scattering_pdf(r, *c, scattered) / pdf; // instrumentation
            bool child_live = live && w.is_finite() && !(w.x == 0.0f && w.y == 0.0f && w.z == 0.0f);
            return emitted + srec->attenuation * c->material->scattering_pdf(r, *c, scattered) *
                                 ray_color(scattered, world, lights, depth + 1, max_depth, background, sky, child_live) / pdf;
        }
        tl_cnt.n_emit_or_miss++;
        return emitted;
    }
    tl_cnt.n_emit_or_miss++;
    return sky ? sky_color(r) : background;
}

// The book-1/2 integrator the legacy Material::scatter methods (still in the reference's API at HEAD,
// src/material.rs:21-28, 85-90, 118-132, 150-175, 215-217, 442-446) were written for.  HEAD has no
// caller for them, so this restates the integrator of the InOneWeekend / TheNextWeek tags in HEAD's
// conventions: depth counted like :126, `emitted + attenuation * ray_color(scattered)`, and either
// the constant background of :124 or the book-1 sky, whose colours sample/inoneweekend.png shows
// ((1-t)*white + t*(0.5,0.7,1.0), t = 0.5*(unit(d).y + 1); its top rows are (220,235,255) = t 0.523).
static Vec3 sky_color(const Ray& r) {
    Vec3 unit_direction = r.direction.unit_vector();
    float t = 0.5f * (unit_direction.y + 1.0f);
    return Vec3::new_const(1.0f) * (1.0f - t) + Vec3(0.5f, 0.7f, 1.0f) * t;
}
static Vec3 ray_color_legacy(const Ray& r, const Arc<Hittable>& world, uint32_t depth, uint32_t max_depth, Vec3 background,
                             bool sky) {
    if (depth > max_depth) return Vec3::new_const(0.0f);
    tl_cnt.rays++;
    tl_cnt.rays_live++;
    if (auto c = world->hit(r, 0.001f, INF)) {
        Vec3 emitted = c->material->emitted(*c, c->u, c->v, c->p);
        if (auto s = c->material->scatter(r, *c)) return emitted + s->first * ray_color_legacy(s->second, world, depth + 1, max_depth, background, sky);
        return emitted;
    }
    return sky ? sky_color(r) : background;
}

// ------------------------------------------------------------------------------------------
// Un-lowering: rebuild the reference's object graph from the flat arrays, so the oracle and
// the GPU see ONE scene instance.  The inverse of the lower() methods of the host front end.
// ------------------------------------------------------------------------------------------
struct Scene {
    std::vector<uint8_t> texels;
    std::vector<Arc<Texture>> textures;
    std::vector<Arc<Material>> materials;
    std::unordered_map<vk_ref, Arc<Hittable>> objects;
    std::unordered_map<const Material*, uint32_t> mat_index;
    Arc<Hittable> world;
    Arc<Hittable> lights; // the Vec<Arc<HittableSS>> of SceneConfig.lights, itself a Hittable
    std::string error;
    const vk_scene_desc* d = nullptr;

    Arc<Hittable> build(vk_ref ref, int depth = 0) {
        auto it = objects.find(ref);
        if (it != objects.end()) return it->second;
        if (depth > 256) throw std::runtime_error("scene graph too deep / cyclic");
        uint32_t i = VK_REF_INDEX(ref);
        Arc<Hittable> h;
        switch (VK_REF_TYPE(ref)) {
        case VK_T_NODE: {
            if (i >= d->n_nodes) throw std::runtime_error("node index out of range");
            const vk_node& n = d->nodes[i];
            auto b = std::make_shared<BVHNode>();
            b->bb.min = Vec3(n.bb_min[0], n.bb_min[1], n.bb_min[2]);
            b->bb.max = Vec3(n.bb_max[0], n.bb_max[1], n.bb_max[2]);
            b->left = build(n.left, depth + 1);
            b->right = n.right == n.left ? b->left : build(n.right, depth + 1);
            h = b;
            break;
        }
        case VK_T_SPHERE: {
            if (i >= d->n_spheres) throw std::runtime_error("sphere index out of range");
            auto s = std::make_shared<Sphere>();
            s->center = Vec3(d->spheres[i].center[0], d->spheres[i].center[1], d->spheres[i].center[2]);
            s->radius = d->spheres[i].radius;
            s->material = materials.at(d->sphere_mat[i]);
            s->id = ref;
            h = s;
            break;
        }
        case VK_T_MSPHERE: {
            if (i >= d->n_mspheres) throw std::runtime_error("msphere index out of range");
            const vk_msphere& m = d->mspheres[i];
            auto s = std::make_shared<MovingSphere>();
            s->center0 = Vec3(m.center0[0], m.center0[1], m.center0[2]);
            s->center1 = Vec3(m.center1[0], m.center1[1], m.center1[2]);
            s->time0 = m.time0; s->time1 = m.time1; s->radius = m.radius;
            s->material = materials.at(m.mat);
            s->id = ref;
            h = s;
            break;
        }
        case VK_T_RECT: {
            if (i >= d->n_rects) throw std::runtime_error("rect index out of range");
            const vk_rect& q = d->rects[i];
            auto r = std::make_shared<Rect>();
            r->c0 = q.c0; r->c1 = q.c1; r->d0 = q.d0; r->d1 = q.d1; r->k = q.k;
            r->axis0 = q.axes & 3; r->axis1 = (q.axes >> 2) & 3; r->axis2 = (q.axes >> 4) & 3;
            r->mat = materials.at(q.mat);
            r->id = ref;
            if (q.axes & VK_RECT_FLIP) h = std::make_shared<FlipFace>(r);
            else h = r;
            break;
        }
        case VK_T_BOX: {
            if (i >= d->n_boxes) throw std::runtime_error("box index out of range");
            const vk_box& b = d->boxes[i];
            h = std::make_shared<Boxy>(Vec3(b.box_min[0], b.box_min[1], b.box_min[2]), Vec3(b.box_max[0], b.box_max[1], b.box_max[2]),
                                       materials.at(b.mat), ref);
            break;
        }
        case VK_T_XFORM: {
            if (i >= d->n_xforms) throw std::runtime_error("xform index out of range");
            const vk_xform& x = d->xforms[i];
            auto child = build(x.child, depth + 1);
            if (x.kind == VK_X_TRANSLATE) {
                auto t = std::make_shared<Translate>();
                t->ptr = child;
                t->offset = Vec3(x.a, x.b, x.c);
                h = t;
            } else if (x.kind == VK_X_FLIP) {
                h = std::make_shared<FlipFace>(child);
            } else if (x.kind <= VK_X_ROTATE_Z) {
                auto r = std::make_shared<Rotate>();
                r->ptr = child;
                r->sin_theta = x.a;
                r->cos_theta = x.b;
                r->kind = x.kind;
                h = r;
            } else
                throw std::runtime_error("bad xform kind");
            break;
        }
        case VK_T_MEDIUM: {
            if (i >= d->n_media) throw std::runtime_error("medium index out of range");
            auto m = std::make_shared<ConstantMedium>();
            m->boundary = build(d->media[i].boundary, depth + 1);
            m->neg_inv_density = d->media[i].neg_inv_density;
            m->phase_function = materials.at(d->media[i].mat);
            m->id = ref;
            h = m;
            break;
        }
        default: throw std::runtime_error("bad hittable reference");
        }
        objects[ref] = h;
        return h;
    }

    void load(const vk_scene_desc* desc) {
        d = desc;
        texels.assign(desc->texels, desc->texels + desc->n_texel_bytes);
        textures.resize(desc->n_textures);
        // children may have larger or smaller indices: create shells first, then wire checkers
        for (uint32_t i = 0; i < desc->n_textures; ++i) {
            const vk_texture& t = desc->textures[i];
            switch (t.type) {
            case VK_TEX_SOLID: textures[i] = std::make_shared<SolidColor>(Vec3(t.rgb[0], t.rgb[1], t.rgb[2])); break;
            case VK_TEX_CHECKER: textures[i] = std::make_shared<Checker>(); break;
            case VK_TEX_IMAGE: {
                auto im = std::make_shared<ImageTexture>();
                im->buf = texels.data() + t.image.texel_offset;
                im->width = t.image.width;
                im->height = t.image.height;
                textures[i] = im;
                break;
            }
            case VK_TEX_NOISE: {
                auto nt = std::make_shared<NoiseTexture>();
                const vk_perlin& p = desc->perlins[t.noise.perlin];
                for (int k = 0; k < 256; ++k) {
                    nt->noise.random_data[k] = Vec3(p.ranvec[k][0], p.ranvec[k][1], p.ranvec[k][2]);
                    nt->noise.perm_x[k] = p.perm_x[k];
                    nt->noise.perm_y[k] = p.perm_y[k];
                    nt->noise.perm_z[k] = p.perm_z[k];
                }
                nt->scale = t.noise.scale;
                textures[i] = nt;
                break;
            }
            default: throw std::runtime_error("bad texture type");
            }
        }
        for (uint32_t i = 0; i < desc->n_textures; ++i)
            if (desc->textures[i].type == VK_TEX_CHECKER) {
                auto c = std::static_pointer_cast<Checker>(textures[i]);
                c->odd = textures.at(desc->textures[i].checker.odd);
                c->even = textures.at(desc->textures[i].checker.even);
            }
        materials.resize(desc->n_materials);
        for (uint32_t i = 0; i < desc->n_materials; ++i) {
            const vk_material& m = desc->materials[i];
            switch (m.type) {
            case VK_M_LAMBERTIAN: { auto x = std::make_shared<Lambertian>(); x->albedo = textures.at(m.tex); materials[i] = x; break; }
            case VK_M_METAL: { auto x = std::make_shared<Metal>(); x->albedo = textures.at(m.tex); x->fuzz = m.param; materials[i] = x; break; }
            case VK_M_DIELECTRIC: { auto x = std::make_shared<Dielectric>(); x->ref_idx = m.param; materials[i] = x; break; }
            case VK_M_DIFFUSE_LIGHT: { auto x = std::make_shared<DiffuseLight>(); x->emit = textures.at(m.tex); materials[i] = x; break; }
            case VK_M_ISOTROPIC: { auto x = std::make_shared<Isotropic>(); x->albedo = textures.at(m.tex); materials[i] = x; break; }
            case VK_M_SPECDIFFUSE: materials[i] = std::make_shared<SpecDiffuse>(); break;
            default: throw std::runtime_error("bad material type");
            }
        }
        for (uint32_t i = 0; i < desc->n_materials; ++i)
            if (desc->materials[i].type == VK_M_SPECDIFFUSE) {
                auto sd = std::static_pointer_cast<SpecDiffuse>(materials[i]);
                sd->specular = materials.at(desc->materials[i].tex);
                sd->diffuse = materials.at(desc->materials[i].aux);
                sd->pct = desc->materials[i].param;
            }
        for (uint32_t i = 0; i < desc->n_materials; ++i) mat_index[materials[i].get()] = i;
        world = build(desc->root);
        auto ll = std::make_shared<ListHittable>();
        for (uint32_t i = 0; i < desc->n_lights; ++i) ll->items.push_back(build(desc->lights[i]));
        lights = ll;
        d = nullptr; // the description is borrowed only for the call
    }
};

static Camera camera_from(const vk_camera* k) {
    Camera c;
    auto v3 = [](const float* p) { return Vec3(p[0], p[1], p[2]); };
    c.origin = v3(k->origin);
    c.lower_left_corner = v3(k->lower_left_corner);
    c.horizontal = v3(k->horizontal);
    c.vertical = v3(k->vertical);
    c.u = v3(k->u);
    c.v = v3(k->v);
    c.w = v3(k->w);
    c.lens_radius = k->lens_radius;
    c.time0 = k->time0;
    c.time1 = k->time1;
    return c;
}

static void write_hit(const std::optional<HitRec>& h, const Scene& sc, vk_hit& o) {
    std::memset(&o, 0, sizeof(o));
    if (!h) return;
    o.prim = h->prim;
    o.face = h->face;
    auto mi = sc.mat_index.find(h->material.get());
    o.mat = mi == sc.mat_index.end() ? 0xFFFFFFFFu : mi->second;
    o.front = h->front ? 1u : 0u;
    o.t = h->t;
    o.p[0] = h->p.x; o.p[1] = h->p.y; o.p[2] = h->p.z;
    o.normal[0] = h->normal.x; o.normal[1] = h->normal.y; o.normal[2] = h->normal.z;
    o.u = h->u;
    o.v = h->v;
}

} // namespace orc

struct orc_scene {
    orc::Scene s;
};
static thread_local std::string g_orc_err;

extern "C" {

const char* orc_last_error(void) { return g_orc_err.c_str(); }

int orc_scene_create(const vk_scene_desc* desc, orc_scene** out) {
    if (!desc || !out || desc->api_version != VK_API_VERSION) {
        g_orc_err = "orc_scene_create: bad argument";
        return VK_ERR_INVALID;
    }
    try {
        auto s = std::make_unique<orc_scene>();
        s->s.load(desc);
        *out = s.release();
        return VK_OK;
    } catch (const std::exception& e) {
        g_orc_err = e.what();
        return VK_ERR_INVALID;
    }
}
void orc_scene_free(orc_scene* s) { delete s; }

int orc_intersect(const orc_scene* s, const vk_ray* rays, size_t n, const float* medium_xi, vk_hit* out) {
    if (!s || !rays || !out) return VK_ERR_INVALID;
    using namespace orc;
#pragma omp parallel
    {
        Rng rng;
        tl_rng = &rng;
#pragma omp for schedule(dynamic, 4096)
        for (long long i = 0; i < (long long)n; ++i) {
            rng.seed(0x1234, (uint64_t)i, 7);
            rng.medium_xi = medium_xi ? medium_xi + (size_t)i * VK_MEDIUM_XI_SLOTS : nullptr;
            std::memset(rng.medium_visits, 0, sizeof(rng.medium_visits));
            const vk_ray& q = rays[i];
            Ray r(Vec3(q.origin[0], q.origin[1], q.origin[2]), Vec3(q.direction[0], q.direction[1], q.direction[2]), q.time);
            auto h = s->s.world->hit(r, q.tmin, q.tmax);
            write_hit(h, s->s, out[i]);
        }
        tl_rng = nullptr;
    }
    return VK_OK;
}

int orc_render(const orc_scene* s, const vk_camera* cam_, const vk_render_params* P, float* out_rgb, float* out_sumsq,
               orc_stats* stats, int n_threads) {
    if (!s || !cam_ || !P || !out_rgb || P->width < 2 || P->height < 2 || P->spp == 0) return VK_ERR_INVALID;
    using namespace orc;
    const Camera cam = camera_from(cam_);
    const uint32_t width = P->width, height = P->height;
    const uint32_t s_begin = P->spp_begin, s_count = P->spp_count ? P->spp_count : P->spp - P->spp_begin;
    const Vec3 background(P->background[0], P->background[1], P->background[2]);
    if (n_threads <= 0) n_threads = omp_get_max_threads();
    Counters total;
    uint64_t dropped = 0;
    auto t0 = std::chrono::steady_clock::now();
#pragma omp parallel num_threads(n_threads)
    {
        Rng rng;
        tl_rng = &rng;
        tl_cnt = Counters();
        uint64_t my_dropped = 0;
        // pixels.par_iter_mut().enumerate().for_each(|(i, pix)| ...)   src/main.rs:181
#pragma omp for schedule(dynamic, 64)
        for (long long i = 0; i < (long long)width * height; ++i) {
            size_t x = (size_t)i % width;
            size_t y = (size_t)i / width;
            Vec3 c = Vec3::new_const(0.0f), c2 = Vec3::new_const(0.0f);
            for (uint32_t sidx = s_begin; sidx < s_begin + s_count; ++sidx) { // :186
                rng.seed(P->seed, (uint64_t)i, sidx); // thread_rng() is unseeded in the reference
                float u = ((float)x + rng.gen_f32()) / (float)(width - 1);
                float v = ((float)y + rng.gen_f32()) / (float)(height - 1);
                Ray ray = cam.get_ray(u, v);
                Vec3 color = (P->flags & VK_FLAG_LEGACY_SCATTER)
                                 ? ray_color_legacy(ray, s->s.world, 1, P->max_depth, background, (P->flags & VK_FLAG_SKY_BACKGROUND) != 0)
                                 : ray_color(ray, s->s.world, s->s.lights, 1, P->max_depth, background,
                                             (P->flags & VK_FLAG_SKY_BACKGROUND) != 0);
                if (color.is_finite()) { // :192-194
                    c = c + color;
                    c2 = c2 + color * color;
                } else
                    my_dropped++;
            }
            c = c / (float)P->spp; // :196 (dropped samples stay in the divisor)
            out_rgb[3 * i + 0] = c.x; out_rgb[3 * i + 1] = c.y; out_rgb[3 * i + 2] = c.z;
            if (out_sumsq) {
                out_sumsq[3 * i + 0] = c2.x; out_sumsq[3 * i + 1] = c2.y; out_sumsq[3 * i + 2] = c2.z;
            }
        }
#pragma omp critical
        {
            const uint64_t* src = reinterpret_cast<const uint64_t*>(&tl_cnt);
            uint64_t* dst = reinterpret_cast<uint64_t*>(&total);
            for (size_t k = 0; k < sizeof(Counters) / sizeof(uint64_t); ++k) dst[k] += src[k];
            dropped += my_dropped;
        }
        tl_rng = nullptr;
    }
    auto t1 = std::chrono::steady_clock::now();
    if (g_scatter_unwrap_panic) {
        g_scatter_unwrap_panic = false;
        return VK_ERR_UNSUPPORTED;
    }
    if (stats) {
        std::memset(stats, 0, sizeof(*stats));
        stats->paths = (uint64_t)width * height * s_count;
        stats->rays = total.rays;
        stats->dropped_samples = dropped;
        stats->n_node = total.n_node; stats->n_sph_rej = total.n_sph_rej; stats->n_sph_acc = total.n_sph_acc;
        stats->n_msph = total.n_msph; stats->n_rect_rej = total.n_rect_rej; stats->n_rect_acc = total.n_rect_acc;
        stats->n_box = total.n_box; stats->n_translate = total.n_translate; stats->n_rotate = total.n_rotate;
        stats->n_medium = total.n_medium; stats->n_texel = total.n_texel; stats->n_perlin = total.n_perlin;
        stats->n_diffuse = total.n_diffuse; stats->n_dielectric = total.n_dielectric; stats->n_metal = total.n_metal;
        stats->n_emit_or_miss = total.n_emit_or_miss; stats->n_light_pdf = total.n_light_pdf;
        stats->rays_live = total.rays_live;
        stats->seconds = std::chrono::duration<double>(t1 - t0).count();
        stats->threads = n_threads;
    }
    return VK_OK;
}

size_t orc_harvest_rays(const orc_scene* s, const vk_camera* cam_, uint32_t width, uint32_t height, uint32_t max_depth,
                        uint64_t seed, size_t max_rays, vk_ray* out) {
    if (!s || !cam_ || !out || width < 2 || height < 2) return 0;
    using namespace orc;
    const Camera cam = camera_from(cam_);
    Rng rng;
    tl_rng = &rng;
    RayTap tap;
    tap.out = out;
    tap.cap = max_rays;
    tl_tap = &tap;
    uint64_t sample = 0;
    while (tap.n < max_rays) {
        size_t before = tap.n;
        for (uint32_t y = 0; y < height && tap.n < max_rays; ++y)
            for (uint32_t x = 0; x < width && tap.n < max_rays; ++x) {
                rng.seed(seed, (uint64_t)y * width + x, sample);
                float u = ((float)x + rng.gen_f32()) / (float)(width - 1);
                float v = ((float)y + rng.gen_f32()) / (float)(height - 1);
                ray_color(cam.get_ray(u, v), s->s.world, s->s.lights, 1, max_depth, Vec3::new_const(0.0f), false);
            }
        ++sample;
        if (tap.n == before) break;
    }
    tl_tap = nullptr;
    tl_rng = nullptr;
    return tap.n;
}

// The oracle's side of vk_eval_batch (include/vecchio_gpu.h): the same record through the restated reference
// code, fed the same 32-bit variates.  The reference draws in program order from one stream, the GPU names its
// draws (xi[0] mixture choice / Schlick test, xi[1..2] the direction, xi[3] light choice, xi[4] SpecDiffuse), so
// the script puts the words in the order this material's code path will ask for them.  Rejection loops
// (random_in_unit_sphere: Metal with fuzz, legacy Isotropic) take their words from the oracle's own stream: the
// GPU samples the same law directly, not the same points.
int orc_eval_batch(const orc_scene* s, vk_eval* recs, size_t n) {
    using namespace orc;
    if (!s || (!recs && n)) return VK_ERR_INVALID;
    Rng rng;
    rng.seed(11, 22, 33);
    tl_rng = &rng;
    auto v3 = [](const float* f) { return Vec3(f[0], f[1], f[2]); };
    auto put3 = [](float* f, Vec3 v) { f[0] = v.x; f[1] = v.y; f[2] = v.z; };
    auto u01 = [](uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); };
    const ListHittable* lights = dynamic_cast<const ListHittable*>(s->s.lights.get());
    int rc = VK_OK;
    for (size_t i = 0; i < n && rc == VK_OK; ++i) {
        vk_eval& e = recs[i];
        std::vector<uint32_t> script;
        if (e.op == VK_EVAL_BOUNCE || e.op == VK_EVAL_BOUNCE_LEGACY) {
            if (e.index >= s->s.materials.size()) { rc = VK_ERR_INVALID; break; }
            const Arc<Material>& mat = s->s.materials[e.index];
            const Material* m = mat.get();
            if (auto sd = dynamic_cast<const SpecDiffuse*>(m)) {
                script.push_back(e.xi[4]);
                m = (u01(e.xi[4]) < sd->pct ? sd->specular : sd->diffuse).get();
            }
            const bool legacy = e.op == VK_EVAL_BOUNCE_LEGACY;
            if (dynamic_cast<const Dielectric*>(m)) script.push_back(e.xi[0]);
            else if (dynamic_cast<const Lambertian*>(m) || (!legacy && dynamic_cast<const Isotropic*>(m))) {
                script.push_back(e.xi[0]);
                if (legacy) script.push_back(e.xi[1]); // Lambertian::random: angle, z
                else if (u01(e.xi[0]) < 0.5f && lights && !lights->items.empty()) { // light branch: choose, then the light's own draws
                    script.push_back(e.xi[3]);
                    const size_t li = (size_t)(((uint64_t)e.xi[3] * (uint64_t)lights->items.size()) >> 32);
                    if (dynamic_cast<const Boxy*>(lights->items[li].get())) script.push_back(e.xi[3] * 0x9E3779B1u); // its side
                    script.push_back(e.xi[1]);
                    script.push_back(e.xi[2]);
                } else {
                    script.push_back(e.xi[1]);
                    script.push_back(e.xi[2]);
                }
            }
            rng.script = script.data();
            rng.script_n = script.size();
            rng.script_pos = 0;
            Ray r(v3(e.ray_o), v3(e.ray_d), e.ray_time);
            HitRec rec(v3(e.p), v3(e.normal), e.t, e.u, e.v, e.front != 0, mat);
            e.alive = 0;
            e.valid = 1;
            Vec3 beta = Vec3::new_const(1.0f), L = Vec3::new_const(0.0f);
            Ray out = r;
            if (!legacy) { // src/main.rs:131-149
                Vec3 emitted = mat->emitted(rec, rec.u, rec.v, rec.p);
                if (auto srec = mat->scatter_with_pdf(r, rec)) {
                    if (srec->specular_ray) {
                        beta = srec->attenuation;
                        out = *srec->specular_ray;
                        e.alive = 1;
                    } else {
                        auto p_important = std::make_shared<HittablePDF>(s->s.lights, rec.p);
                        MixturePDF p(p_important, 0.5f, srec->pdf, 0.5f);
                        Ray scattered(rec.p, p.generate(), r.time);
                        float pdf = p.value(scattered.direction);
                        beta = srec->attenuation * mat->scattering_pdf(r, rec, scattered) / pdf;
                        L = emitted;
                        out = scattered;
                        e.alive = 1;
                        e.value = pdf;
                        if (!beta.is_finite()) e.valid = 0;
                    }
                } else
                    L = emitted;
            } else { // ray_color_legacy
                g_scatter_unwrap_panic = false;
                L = mat->emitted(rec, rec.u, rec.v, rec.p);
                if (auto sc = mat->scatter(r, rec)) {
                    beta = sc->first;
                    out = sc->second;
                    e.alive = 1;
                }
                if (g_scatter_unwrap_panic) e.valid = 0;
            }
            rng.script = nullptr;
            put3(e.out_o, out.origin);
            put3(e.out_d, out.direction);
            e.out_time = out.time;
            put3(e.beta, beta);
            put3(e.L, L);
        } else if (e.op == VK_EVAL_TEXTURE) {
            if (e.index >= s->s.textures.size()) { rc = VK_ERR_INVALID; break; }
            put3(e.beta, s->s.textures[e.index]->value(e.u, e.v, v3(e.p)));
        } else if (e.op == VK_EVAL_LIGHTS_PDF) {
            e.value = s->s.lights->pdf_value(v3(e.p), v3(e.dir));
        } else if (e.op == VK_EVAL_LIGHT_RANDOM) {
            if (!lights || e.index >= lights->items.size()) { rc = VK_ERR_INVALID; break; }
            const Hittable* l = lights->items[e.index].get();
            if (dynamic_cast<const Boxy*>(l)) script.push_back(e.xi[2]); // Boxy::random: choose a side, then the side's draws
            script.push_back(e.xi[0]);
            script.push_back(e.xi[1]);
            rng.script = script.data();
            rng.script_n = script.size();
            rng.script_pos = 0;
            put3(e.out_d, l->random(v3(e.p)));
            rng.script = nullptr;
        } else
            rc = VK_ERR_INVALID;
    }
    tl_rng = nullptr;
    return rc;
}

int orc_kat(const orc_scene* s, const char* name, const float* in, int n_in, float* out, int n_out) {
    using namespace orc;
    std::string k(name ? name : "");
    auto v3 = [&](int o) { return Vec3(in[o], in[o + 1], in[o + 2]); };
    auto put3 = [&](int o, Vec3 v) { out[o] = v.x; out[o + 1] = v.y; out[o + 2] = v.z; };
    Rng rng;
    rng.seed(1, 2, 3);
    tl_rng = &rng;
    int ret = -1;
    if (k == "spherical" && n_in >= 3 && n_out >= 2) {
        spherical(v3(0), out[0], out[1]);
        ret = 2;
    } else if (k == "reflect" && n_in >= 6 && n_out >= 3) {
        put3(0, reflect(v3(0), v3(3)));
        ret = 3;
    } else if (k == "refract" && n_in >= 7 && n_out >= 3) {
        put3(0, refract(v3(0), v3(3), in[6]));
        ret = 3;
    } else if (k == "schlick" && n_in >= 2 && n_out >= 1) {
        out[0] = schlick(in[0], in[1]);
        ret = 1;
    } else if (k == "onb" && n_in >= 3 && n_out >= 9) {
        ONB o = ONB::new_from_w(v3(0));
        put3(0, o.u); put3(3, o.v); put3(6, o.w);
        ret = 9;
    } else if (k == "sky_color" && n_in >= 3 && n_out >= 3) { // direction -> book-1 sky
        put3(0, sky_color(Ray(Vec3::new_const(0.0f), v3(0))));
        ret = 3;
    } else if (k == "aabb_hit" && n_in >= 14 && n_out >= 1) { // min3 max3 o3 d3 tmin tmax
        AxisBB bb{v3(0), v3(3)};
        out[0] = bb.hit(Ray(v3(6), v3(9)), in[12], in[13]) ? 1.0f : 0.0f;
        ret = 1;
    } else if (k == "sphere_hit" && n_in >= 12 && n_out >= 10) { // c3 r o3 d3 tmin tmax -> hit t p3 n3 front u v
        Sphere sp;
        sp.center = v3(0);
        sp.radius = in[3];
        sp.material = std::make_shared<Dielectric>();
        auto h = sp.hit(Ray(v3(4), v3(7)), in[10], in[11]);
        out[0] = h ? 1.0f : 0.0f;
        if (h) {
            out[1] = h->t; put3(2, h->p); put3(5, h->normal);
            out[8] = h->front ? 1.0f : 0.0f; out[9] = h->u;
            if (n_out >= 11) out[10] = h->v;
        }
        ret = 11;
    } else if (k == "rect_pdf_value" && n_in >= 14 && n_out >= 1) { // c0 c1 d0 d1 k a0 a1 a2 o3 v3
        Rect r;
        r.c0 = in[0]; r.c1 = in[1]; r.d0 = in[2]; r.d1 = in[3]; r.k = in[4];
        r.axis0 = (size_t)in[5]; r.axis1 = (size_t)in[6]; r.axis2 = (size_t)in[7];
        r.mat = std::make_shared<Dielectric>();
        out[0] = r.pdf_value(v3(8), v3(11));
        ret = 1;
    } else if (k == "to_color" && n_in >= 3 && n_out >= 3) {
        uint32_t c[3];
        to_color(v3(0), c);
        out[0] = (float)c[0]; out[1] = (float)c[1]; out[2] = (float)c[2];
        ret = 3;
    } else if (k == "texture_value" && s && n_in >= 6 && n_out >= 3) { // tex_index u v p3
        size_t ti = (size_t)in[0];
        if (ti < s->s.textures.size()) {
            put3(0, s->s.textures[ti]->value(in[1], in[2], v3(3)));
            ret = 3;
        }
    } else if (k == "camera_get_ray" && n_in >= 26 && n_out >= 7) { // 24 camera floats, s, t
        vk_camera c;
        std::memcpy(&c, in, sizeof(c));
        Ray r = camera_from(&c).get_ray(in[24], in[25]);
        put3(0, r.origin); put3(3, r.direction); out[6] = r.time;
        ret = 7;
    } else if (k == "cosine_pdf_value" && n_in >= 6 && n_out >= 1) {
        out[0] = CosinePDF(v3(0)).value(v3(3));
        ret = 1;
    } else if (k == "material_scatter" && n_in >= 19 && n_out >= 12) {
        // type(0 Lambertian 1 Metal 2 Dielectric 4 Isotropic) albedo3 param | ray o3 d3 time | hit p3 n3 front  ->
        // n_out/12 draws of scatter_with_pdf: {scattered?, specular?, ray o3 d3 time, attenuation3, pdf.value(d) or 0}
        auto tex = std::make_shared<SolidColor>(v3(1));
        Arc<Material> m;
        const int type = (int)in[0];
        if (type == 0) { auto x = std::make_shared<Lambertian>(); x->albedo = tex; m = x; }
        else if (type == 1) { auto x = std::make_shared<Metal>(); x->albedo = tex; x->fuzz = in[4]; m = x; }
        else if (type == 2) { auto x = std::make_shared<Dielectric>(); x->ref_idx = in[4]; m = x; }
        else if (type == 4) { auto x = std::make_shared<Isotropic>(); x->albedo = tex; m = x; }
        if (m) {
            Ray r(v3(5), v3(8), in[11]);
            HitRec rec(v3(12), v3(15), 1.0f, 0.0f, 0.0f, in[18] != 0.0f, m);
            Vec3 probe = v3(19 <= n_in - 3 ? 19 : 15); // direction at which the returned pdf is evaluated (default: the normal)
            ret = 0;
            for (int i = 0; i + 12 <= n_out; i += 12, ret += 12) {
                float* o = out + i;
                for (int j = 0; j < 12; j++) o[j] = 0.0f;
                auto srec = m->scatter_with_pdf(r, rec);
                if (!srec) continue;
                o[0] = 1.0f;
                if (srec->specular_ray) {
                    o[1] = 1.0f;
                    put3(i + 2, srec->specular_ray->origin); put3(i + 5, srec->specular_ray->direction);
                    o[8] = srec->specular_ray->time;
                } else
                    o[8] = srec->pdf->value(probe);
                put3(i + 9, srec->attenuation);
            }
        }
    } else if (k == "sphere_pdf_value" && n_in >= 10 && n_out >= 1) { // c3 r o3 d3
        Sphere sp;
        sp.center = v3(0);
        sp.radius = in[3];
        sp.material = std::make_shared<Dielectric>();
        out[0] = sp.pdf_value(v3(4), v3(7));
        ret = 1;
    } else if (k == "sphere_random" && n_in >= 7 && n_out >= 3) { // c3 r o3 -> n_out/3 draws of Sphere::random
        Sphere sp;
        sp.center = v3(0);
        sp.radius = in[3];
        sp.material = std::make_shared<Dielectric>();
        ret = 0;
        for (int i = 0; i + 3 <= n_out; i += 3, ret += 3) put3(i, sp.random(v3(4)));
    } else if (k == "box_pdf_value" && n_in >= 12 && n_out >= 1) { // p0 p1 o3 v3
        Boxy bx(v3(0), v3(3), std::make_shared<Dielectric>(), VK_REF_NONE);
        out[0] = bx.pdf_value(v3(6), v3(9));
        ret = 1;
    } else if (k == "box_random" && n_in >= 9 && n_out >= 3) { // p0 p1 o3 -> n_out/3 draws of Boxy::random
        Boxy bx(v3(0), v3(3), std::make_shared<Dielectric>(), VK_REF_NONE);
        ret = 0;
        for (int i = 0; i + 3 <= n_out; i += 3, ret += 3) put3(i, bx.random(v3(6)));
    }
    tl_rng = nullptr;
    return ret;
}

} // extern "C"
