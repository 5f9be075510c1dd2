// scene.cpp -- the scene builders of the reference (src/scene.rs) on the C++ host front end,
// plus the two BASELINE.json configurations the reference does not ship (Cornell smoke, the
// 1M-sphere stress scene), authored with the same API.  Host-only: these feed the hot path.
#include "vecchio.hpp"

namespace vecchio {

namespace {

template <class T, class... A> Arc<T> arc(A&&... a) { return std::make_shared<T>(std::forward<A>(a)...); }
Arc<TextureSS> solid(float r, float g, float b) { return arc<SolidColor>(Vec3(r, g, b)); }
Arc<MaterialSS> lambert(float r, float g, float b) { return arc<Lambertian>(solid(r, g, b)); }
Arc<HittableSS> rect(Rect r) { return std::make_shared<Rect>(std::move(r)); }
Arc<HittableSS> flip(Arc<HittableSS> h) { return arc<FlipFace>(std::move(h)); }

// FixedCamera (src/scene.rs:24-46)
struct FixedCamera : CameraIter {
    Camera cam;
    bool called = false;
    explicit FixedCamera(Camera c) : cam(c) {}
    std::optional<Camera> next() override {
        if (called) return std::nullopt;
        called = true;
        return cam;
    }
};

// RotatingCamera (src/scene.rs:48-91)
struct RotatingCamera : CameraIter {
    Vec3 lookat, vup;
    float vfov, aspect_ratio, aperture, focus_dist, time0, time1, height, angle, radius, incr, limit;
    std::optional<Camera> next() override {
        if (angle > limit) return std::nullopt;
        float look_x = radius * std::cos(to_radians(angle));
        float look_z = radius * std::sin(to_radians(angle));
        Camera cam = Camera::make(Vec3(look_x, height, look_z), lookat, vup, vfov, aspect_ratio, aperture,
                                  focus_dist, time0, time1);
        angle += incr;
        return cam;
    }
};

std::unique_ptr<CameraIter> fixed(Vec3 from, Vec3 at, float vfov, float aspect) {
    return std::make_unique<FixedCamera>(Camera::make(from, at, Vec3(0, 1, 0), vfov, aspect, 0.0f, 10.0f, 0.0f, 1.0f));
}
std::unique_ptr<CameraIter> rotating(Vec3 at, float vfov, float aspect, float height, float angle, float radius,
                                     float incr, float limit) {
    auto c = std::make_unique<RotatingCamera>();
    c->lookat = at;
    c->vup = Vec3(0, 1, 0);
    c->vfov = vfov;
    c->aspect_ratio = aspect;
    c->aperture = 0.0f;
    c->focus_dist = 10.0f;
    c->time0 = 0.0f;
    c->time1 = 1.0f;
    c->height = height;
    c->angle = angle;
    c->radius = radius;
    c->incr = incr;
    c->limit = limit;
    return c;
}

// the square sky light shared by balls_demo / perlin_demo (src/scene.rs:129-140, 303-314)
void push_sky_light(SceneConfig& s, float half, float y, Vec3 emit) {
    auto shape = rect(Rect::XZRect(-half, half, -half, half, y, arc<DiffuseLight>(arc<SolidColor>(emit))));
    s.world.push_back(flip(shape));
    s.lights.push_back(shape);
}

// the 80 / 15 / 5 material rule of src/scene.rs:194-215
Arc<MaterialSS> random_small_sphere_material(float choose_mat) {
    auto& rng = thread_rng();
    if (choose_mat < 0.8f) {
        Vec3 albedo = Vec3::random() * Vec3::random();
        return arc<Lambertian>(arc<SolidColor>(albedo));
    } else if (choose_mat < 0.95f) {
        auto albedo = arc<SolidColor>(Vec3::random_range(0.5f, 1.0f));
        float fuzz = rng.gen_range(0.0f, 0.5f);
        return arc<Metal>(albedo, fuzz);
    }
    return arc<Dielectric>(1.5f);
}

// Bowser (src/scene.rs:340-549): a user-defined Hittable that delegates to an inner BVH.
struct Bowser : Hittable {
    Arc<HittableSS> parts;
    Bowser(float x, float y, float z) {
        std::vector<Arc<HittableSS>> w;
        const float yb = y - 1.875f, zb = z + 4.5f;
        auto img = [](const char* p) { return arc<Lambertian>(arc<ImageTexture>(p)); };
        // face, top, back, two sides, bottom (:347-412)
        w.push_back(rect(Rect::XYRect(x - 2.0f, x + 2.0f, yb + 1.0f, yb + 4.0f, zb - 3.0f, img("assets/bowser_face.png"))));
        w.push_back(rect(Rect::XZRect(x - 2.0f, x + 2.0f, zb - 6.0f, zb - 3.0f, yb + 4.0f, img("assets/bowser_top.png"))));
        w.push_back(rect(Rect::XYRect(x - 2.0f, x + 2.0f, yb + 1.0f, yb + 4.0f, zb - 6.0f, img("assets/bowser_back.png"))));
        w.push_back(rect(Rect::YZRect(yb + 1.0f, yb + 4.0f, zb - 6.0f, zb - 3.0f, x - 2.0f, img("assets/bowser_side.png"))));
        w.push_back(rect(Rect::YZRect(yb + 1.0f, yb + 4.0f, zb - 6.0f, zb - 3.0f, x + 2.0f, img("assets/bowser_side.png"))));
        auto grey = lambert(0.278f, 0.387f, 0.438f);
        w.push_back(rect(Rect::XZRect(x - 2.0f, x + 2.0f, zb - 6.0f, zb - 3.0f, yb + 1.0f, grey)));
        struct B { float x0, y0, z0, x1, y1, z1; };
        auto boxes = [&](std::initializer_list<B> bs, Arc<MaterialSS> m) {
            for (const B& b : bs)
                w.push_back(arc<Boxy>(Vec3(x + b.x0, yb + b.y0, zb - b.z0), Vec3(x + b.x1, yb + b.y1, zb - b.z1), m));
        };
        // feet (:413-433)
        boxes({{-1.5f, 0.5f, 4.75f, -0.5f, 1.0f, 4.25f}, {0.5f, 0.5f, 4.75f, 1.5f, 1.0f, 4.25f},
               {-1.5f, 0.25f, 4.75f, -0.5f, 0.5f, 3.5f}, {0.5f, 0.25f, 4.75f, 1.5f, 0.5f, 3.5f}}, grey);
        // arms (:434-467)
        boxes({{-2.25f, 1.75f, 4.65f, -2.00f, 2.75f, 4.35f}, {-2.50f, 1.75f, 4.65f, -2.25f, 2.50f, 4.35f},
               {-2.75f, 1.75f, 4.65f, -2.50f, 2.25f, 4.35f}, {2.00f, 1.75f, 4.65f, 2.25f, 2.75f, 4.35f},
               {2.25f, 1.75f, 4.65f, 2.50f, 2.50f, 4.35f}, {2.50f, 1.75f, 4.65f, 2.75f, 2.25f, 4.35f}},
              lambert(0.4f, 0.2f, 0.1f));
        // face rim (:468-491) and rear ports (:493-534)
        boxes({{-2.0f, 3.875f, 3.00f, 2.0f, 4.00f, 2.875f}, {-2.0f, 1.0f, 3.00f, 2.0f, 1.125f, 2.875f},
               {-2.0f, 1.125f, 3.00f, -1.875f, 3.875f, 2.875f}, {1.875f, 1.125f, 3.00f, 2.0f, 3.875f, 2.875f},
               {-1.875f, 1.625f, 6.125f, -0.875f, 1.75f, 6.0f}, {-1.875f, 1.125f, 6.125f, -0.875f, 1.25f, 6.0f},
               {-1.875f, 1.25f, 6.125f, -1.750f, 1.625f, 6.0f}, {-1.0f, 1.25f, 6.125f, -0.875f, 1.625f, 6.0f},
               {0.875f, 1.625f, 6.125f, 1.875f, 1.75f, 6.0f}, {0.875f, 1.125f, 6.125f, 1.875f, 1.25f, 6.0f},
               {1.750f, 1.25f, 6.125f, 1.875f, 1.625f, 6.0f}, {0.875f, 1.25f, 6.125f, 1.0f, 1.625f, 6.0f}},
              lambert(0.601f, 0.687f, 0.723f));
        parts = BVHNode::make(w);
    }
    std::optional<AxisBB> bounding_box(float t0, float t1) const override { return parts->bounding_box(t0, t1); }
    vk_ref lower(Lowering& L) const override { return L.hittable(parts); } // delegate, like hit() does
};

// the five Cornell walls (src/scene.rs:645-672)
void push_cornell_walls(SceneConfig& s, Arc<MaterialSS> white) {
    s.world.push_back(flip(rect(Rect::YZRect(0, 555, 0, 555, 555, lambert(0.12f, 0.45f, 0.15f)))));
    s.world.push_back(rect(Rect::YZRect(0, 555, 0, 555, 0, lambert(0.65f, 0.05f, 0.05f))));
    s.world.push_back(flip(rect(Rect::XZRect(0, 555, 0, 555, 0, white))));
    s.world.push_back(rect(Rect::XZRect(0, 555, 0, 555, 555, white)));
    s.world.push_back(flip(rect(Rect::XYRect(0, 555, 0, 555, 555, white))));
}
Arc<HittableSS> cornell_block(Vec3 size, float angle, Vec3 offset, Arc<MaterialSS> m) {
    return arc<Translate>(arc<RotateY>(arc<Boxy>(Vec3::new_const(0.0f), size, std::move(m)), angle), offset);
}

} // namespace

// src/scene.rs:93-165
SceneConfig balls_demo() {
    SceneConfig s;
    s.world.push_back(arc<Sphere>(Vec3(0, 0, -1), 0.5f, lambert(0.1f, 0.2f, 0.5f)));
    s.world.push_back(arc<Sphere>(Vec3(0, -100.5f, -1), 100.0f, lambert(0.8f, 0.8f, 0.8f)));
    s.world.push_back(arc<Sphere>(Vec3(1, 0, -1), 0.5f, arc<Metal>(solid(0.8f, 0.6f, 0.2f), 0.3f)));
    s.world.push_back(arc<Sphere>(Vec3(-1, 0, -1), 0.5f, arc<Dielectric>(1.5f)));
    s.world.push_back(arc<Sphere>(Vec3(-1, 0, -1), -0.45f, arc<Dielectric>(1.5f)));
    push_sky_light(s, 6.0f, 8.0f, Vec3::new_const(4.0f));
    s.aspect_ratio = 16.0f / 9.0f;
    s.cam_iter = fixed(Vec3(0, 2, 10), Vec3(0, 1, 0), 40.0f, s.aspect_ratio);
    return s;
}

// Authored with the reference's API to exercise the surface no shipped scene touches (SURVEY 8f rank
// 4): a SpecDiffuse material (src/material.rs:467-488), and a Sphere and a Boxy in the light list
// (cone sampling with the reference's (1-z*z) quirk, src/hittable.rs:104-134; Boxy sides, :371-377).
SceneConfig api_surface_demo() {
    SceneConfig s;
    s.world.push_back(arc<Sphere>(Vec3(0, -100.5f, -1), 100.0f, lambert(0.8f, 0.8f, 0.8f)));
    s.world.push_back(arc<Sphere>(Vec3(0, 0, -1), 0.5f,
                                  arc<SpecDiffuse>(arc<Metal>(solid(0.9f, 0.9f, 0.9f), 0.05f), lambert(0.1f, 0.2f, 0.5f), 0.25f)));
    s.world.push_back(arc<Sphere>(Vec3(1, 0, -1), 0.5f, arc<Metal>(solid(0.8f, 0.6f, 0.2f), 0.3f)));
    s.world.push_back(arc<Sphere>(Vec3(-1, 0, -1), 0.5f, arc<Dielectric>(1.5f)));
    auto ball_light = arc<Sphere>(Vec3(-2.2f, 1.6f, -0.5f), 0.4f, arc<DiffuseLight>(solid(6.0f, 5.0f, 4.0f)));
    s.world.push_back(ball_light);
    s.lights.push_back(ball_light);
    auto box_light = arc<Boxy>(Vec3(1.8f, 1.2f, -1.6f), Vec3(2.4f, 1.6f, -1.0f), arc<DiffuseLight>(solid(3.0f, 4.0f, 6.0f)));
    s.world.push_back(box_light);
    s.lights.push_back(box_light);
    push_sky_light(s, 3.0f, 6.0f, Vec3::new_const(2.0f));
    s.aspect_ratio = 16.0f / 9.0f;
    s.cam_iter = fixed(Vec3(0, 2, 10), Vec3(0, 1, 0), 40.0f, s.aspect_ratio);
    return s;
}

// A furnace, authored with the reference's constructors for its closed-form answer: one convex object inside a
// uniformly emitting room (six DiffuseLight rects at +-40, those on the + side in a FlipFace so that the inside
// is their front, as the Cornell light is built, src/scene.rs:660-668; emission E).  A Sphere of negative radius
// would not do: its bounding box is inverted (src/hittable.rs:97-102) and the BVH would only find it through the
// other object's box.  Every direction leaving the object ends on the room, so the object's radiance is exactly
// albedo * E for a Lambertian (`kind` 0) whatever the sampling strategy, albedo * E for a fuzz-0 Metal (1), and E
// for a Dielectric (2, up to the depth cap) and, in expectation, for a white ConstantMedium (3); pixels beside
// the object show E.  Kind 4 is kind 0 with the room 1000 times as bright, E = (800, 600, 400): the samples beside the
// sphere lie above 255, where the squares behind adaptive sampling's stopping rule clamp, and the sphere's straddle it
// in R and B.  The light list holds a rect OUTSIDE
// the room and not in the world -- the reference keeps lights in their own list (src/main.rs:169) and
// `pdf_value` tests only the light's own geometry -- so the mixture estimator must weight light-sampled
// directions correctly although they never reach that rect.
SceneConfig furnace_demo(uint32_t kind) {
    SceneConfig s;
    auto glow = arc<DiffuseLight>(kind == 4 ? solid(800.0f, 600.0f, 400.0f) : solid(0.8f, 0.6f, 0.4f));
    const float L = 40.0f;
    s.world.push_back(rect(Rect::XYRect(-L, L, -L, L, -L, glow)));
    s.world.push_back(flip(rect(Rect::XYRect(-L, L, -L, L, L, glow))));
    s.world.push_back(rect(Rect::XZRect(-L, L, -L, L, -L, glow)));
    s.world.push_back(flip(rect(Rect::XZRect(-L, L, -L, L, L, glow))));
    s.world.push_back(rect(Rect::YZRect(-L, L, -L, L, -L, glow)));
    s.world.push_back(flip(rect(Rect::YZRect(-L, L, -L, L, L, glow))));
    Arc<MaterialSS> m = kind == 1   ? Arc<MaterialSS>(arc<Metal>(solid(0.7f, 0.6f, 0.5f), 0.0f))
                        : kind == 2 ? Arc<MaterialSS>(arc<Dielectric>(1.5f))
                                    : lambert(0.5f, 0.25f, 0.75f);
    if (kind == 3) // a white medium conserves energy: E in expectation however often the path scatters inside
        s.world.push_back(arc<ConstantMedium>(arc<Sphere>(Vec3(0, 0, 0), 2.0f, m), 0.8f, solid(1, 1, 1)));
    else
        s.world.push_back(arc<Sphere>(Vec3(0, 0, 0), 2.0f, m));
    s.lights.push_back(rect(Rect::XZRect(-6, 6, -6, 6, 70, arc<DiffuseLight>(solid(1, 1, 1)))));
    s.aspect_ratio = 1.0f;
    s.cam_iter = fixed(Vec3(0, 0, 12), Vec3(0, 0, 0), 40.0f, s.aspect_ratio);
    return s;
}

// src/scene.rs:167-284; `with_light` = false gives the book-1 cover as it was before the light was
// added (sample/inoneweekend.png): lit by the sky only, so it needs the legacy integrator
// (VK_FLAG_LEGACY_SCATTER | VK_FLAG_SKY_BACKGROUND) -- HEAD panics on its empty light list.
//
// `book1` = the scene as the book's first volume ends and as sample/inoneweekend.png shows it: grey ground
// (0.5, 0.5, 0.5), a brown Lambertian (0.4, 0.2, 0.1) where HEAD has the earth, no light, and the book's
// fixed camera: lookfrom (13, 2, 3), lookat origin, vfov 20, aperture 0.1, focus 10.  HEAD's scene.rs no
// longer holds this variant; it is authored here with the reference's constructors so that the legacy
// integrator can be checked against the published render.
static SceneConfig random_spheres(bool with_light, bool book1 = false) {
    SceneConfig s;
    auto checker = arc<Checker>(solid(0.1f, 0.1f, 0.1f), solid(0.9f, 0.9f, 0.9f));
    s.world.push_back(arc<Sphere>(Vec3(0, -1000, 0), 1000.0f,
                                  book1 ? lambert(0.5f, 0.5f, 0.5f) : Arc<MaterialSS>(arc<Lambertian>(checker))));

    auto& rng = thread_rng();
    for (int a = -11; a < 11; ++a)
        for (int b = -11; b < 11; ++b) {
            float choose_mat = rng.gen_f32();
            float cx = (float)a + 0.9f * rng.gen_f32();
            float cz = (float)b + 0.9f * rng.gen_f32();
            Vec3 center(cx, 0.2f, cz);
            if ((center - Vec3(4.0f, 0.2f, 0.0f)).length() > 0.9f)
                s.world.push_back(arc<Sphere>(center, 0.2f, random_small_sphere_material(choose_mat)));
        }

    s.world.push_back(arc<Sphere>(Vec3(0, 1, 0), 1.0f, arc<Dielectric>(1.5f)));
    s.world.push_back(arc<Sphere>(Vec3(-4, 1, 0), 1.0f,
                                  book1 ? lambert(0.4f, 0.2f, 0.1f)
                                        : Arc<MaterialSS>(arc<Lambertian>(arc<ImageTexture>("assets/earthmap.png")))));
    s.world.push_back(arc<Sphere>(Vec3(4, 1, 0), 1.0f, arc<Metal>(solid(0.7f, 0.6f, 0.5f), 0.0f)));

    if (with_light) push_sky_light(s, 11.0f, 8.0f, Vec3(1.0f, 0.77f, 0.56f) * 2.0f);

    s.aspect_ratio = 16.0f / 9.0f;
    if (book1)
        s.cam_iter = std::make_unique<FixedCamera>(
            Camera::make(Vec3(13, 2, 3), Vec3(0, 0, 0), Vec3(0, 1, 0), 20.0f, s.aspect_ratio, 0.1f, 10.0f, 0.0f, 1.0f));
    else
        s.cam_iter = rotating(Vec3(0, 1.5f, 0), 20.0f, s.aspect_ratio, 2.5f, 25.0f, 20.0f, 0.5f, 360.0f);
    return s;
}
SceneConfig random_spheres_demo() { return random_spheres(true); }
SceneConfig random_spheres_cover() { return random_spheres(false); }
SceneConfig book1_cover() { return random_spheres(false, true); }

// src/scene.rs:286-338
SceneConfig perlin_demo() {
    SceneConfig s;
    auto pertext = arc<Lambertian>(arc<NoiseTexture>(2.0f));
    s.world.push_back(arc<Sphere>(Vec3(0, -1000, 0), 1000.0f, pertext));
    s.world.push_back(arc<Sphere>(Vec3(0, 2, 0), 2.0f, pertext));
    push_sky_light(s, 6.0f, 8.0f, Vec3::new_const(4.0f));
    s.aspect_ratio = 16.0f / 9.0f;
    s.cam_iter = fixed(Vec3(0, 2, 10), Vec3(0, 1, 0), 40.0f, s.aspect_ratio);
    return s;
}

// src/scene.rs:551-628
SceneConfig bowser_demo() {
    SceneConfig s;
    auto checker = arc<Checker>(solid(0.1f, 0.1f, 0.1f), solid(0.9f, 0.9f, 0.9f));
    s.world.push_back(arc<Sphere>(Vec3(0, -1000, 0), 1000.0f, arc<Lambertian>(checker)));
    s.world.push_back(arc<Translate>(
        arc<RotateX>(arc<RotateY>(arc<RotateZ>(arc<Bowser>(0.0f, 0.0f, 0.0f), 0.0f), 0.0f), 0.0f),
        Vec3(0.0f, 1.625f, -4.5f)));
    auto light_shape =
        rect(Rect::XYRect(-2, 2, 1, 4, 3, arc<DiffuseLight>(arc<ImageTexture>("assets/twitter.png"))));
    s.world.push_back(flip(light_shape));
    s.lights.push_back(light_shape);
    s.aspect_ratio = 16.0f / 9.0f;
    s.cam_iter = rotating(Vec3(0, 2, 0), 20.0f, s.aspect_ratio, 2.5f, -35.0f, 20.0f, 0.5f, 360.0f - 35.0f);
    return s;
}

// src/scene.rs:630-730
SceneConfig cornell_box() {
    SceneConfig s;
    auto white = lambert(0.73f, 0.73f, 0.73f);
    push_cornell_walls(s, white);
    s.world.push_back(cornell_block(Vec3(165, 330, 165), 15.0f, Vec3(265, 0, 295), white));
    s.world.push_back(arc<Sphere>(Vec3(190, 90, 190), 90.0f, arc<Dielectric>(1.5f)));
    auto light_shape = rect(Rect::XZRect(213, 343, 227, 332, 554, arc<DiffuseLight>(solid(15, 15, 15))));
    s.world.push_back(flip(light_shape));
    s.lights.push_back(light_shape);
    s.aspect_ratio = 1.0f;
    s.cam_iter = fixed(Vec3(278, 278, -800), Vec3(278, 278, 0), 40.0f, s.aspect_ratio);
    return s;
}

// BASELINE.json config 3 (book 2 "Cornell smoke"), SURVEY.md 8(d).  Not in src/scene.rs.
SceneConfig cornell_smoke() {
    SceneConfig s;
    auto white = lambert(0.73f, 0.73f, 0.73f);
    push_cornell_walls(s, white);
    auto light_shape = rect(Rect::XZRect(113, 443, 127, 432, 554, arc<DiffuseLight>(solid(7, 7, 7))));
    s.world.push_back(flip(light_shape));
    s.lights.push_back(light_shape);
    s.world.push_back(arc<ConstantMedium>(cornell_block(Vec3(165, 330, 165), 15.0f, Vec3(265, 0, 295), white), 0.01f,
                                          solid(0, 0, 0)));
    s.world.push_back(arc<ConstantMedium>(cornell_block(Vec3(165, 165, 165), -18.0f, Vec3(130, 0, 65), white), 0.01f,
                                          solid(1, 1, 1)));
    s.aspect_ratio = 1.0f;
    s.cam_iter = fixed(Vec3(278, 278, -800), Vec3(278, 278, 0), 40.0f, s.aspect_ratio);
    return s;
}

// src/scene.rs:732-874
SceneConfig final_scene() {
    SceneConfig s;
    auto& rng = thread_rng();
    std::vector<Arc<HittableSS>> boxes1;
    auto ground = lambert(0.48f, 0.83f, 0.53f);
    const int BOXES_PER_SIDE = 20;
    for (int i = 0; i < BOXES_PER_SIDE; ++i)
        for (int j = 0; j < BOXES_PER_SIDE; ++j) {
            float w = 100.0f;
            float x0 = -1000.0f + (float)i * w, z0 = -1000.0f + (float)j * w, y0 = 0.0f;
            float x1 = x0 + w, z1 = z0 + w, y1 = rng.gen_range(1.0f, 101.0f);
            boxes1.push_back(arc<Boxy>(Vec3(x0, y0, z0), Vec3(x1, y1, z1), ground));
        }
    s.world.push_back(BVHNode::make(boxes1));

    auto light_shape = rect(Rect::XZRect(123, 423, 147, 412, 554, arc<DiffuseLight>(arc<SolidColor>(Vec3::new_const(7.0f)))));
    s.world.push_back(flip(light_shape));
    s.lights.push_back(light_shape);

    Vec3 center1(400, 400, 200), center2 = center1 + Vec3(30, 0, 0);
    s.world.push_back(arc<MovingSphere>(center1, center2, 0.0f, 1.0f, 50.0f, lambert(0.7f, 0.3f, 0.1f)));
    s.world.push_back(arc<Sphere>(Vec3(260, 150, 45), 50.0f, arc<Dielectric>(1.5f)));
    s.world.push_back(arc<Sphere>(Vec3(0, 150, 145), 50.0f, arc<Metal>(solid(0.8f, 0.8f, 0.9f), 10.0f)));

    auto boundary1 = arc<Sphere>(Vec3(360, 150, 145), 70.0f, arc<Dielectric>(1.5f));
    s.world.push_back(boundary1);
    s.world.push_back(arc<ConstantMedium>(boundary1, 0.2f, solid(0.2f, 0.4f, 0.9f)));
    auto boundary2 = arc<Sphere>(Vec3::new_const(0.0f), 5000.0f, arc<Dielectric>(1.5f));
    s.world.push_back(arc<ConstantMedium>(boundary2, 0.0001f, arc<SolidColor>(Vec3::new_const(1.0f))));

    s.world.push_back(arc<Sphere>(Vec3(400, 200, 400), 100.0f, arc<Lambertian>(arc<ImageTexture>("assets/earthmap.png"))));
    s.world.push_back(arc<Sphere>(Vec3(220, 280, 300), 80.0f, arc<Lambertian>(arc<NoiseTexture>(0.1f))));

    std::vector<Arc<HittableSS>> boxes2;
    auto white = arc<Lambertian>(arc<SolidColor>(Vec3::new_const(0.73f)));
    for (int i = 0; i < 1000; ++i) boxes2.push_back(arc<Sphere>(Vec3::random_range(0.0f, 165.0f), 10.0f, white));
    s.world.push_back(arc<Translate>(arc<RotateY>(BVHNode::make(boxes2), 15.0f), Vec3(-100, 270, 395)));

    s.aspect_ratio = 1.0f;
    s.cam_iter = fixed(Vec3(478, 278, -600), Vec3(278, 278, 0), 40.0f, s.aspect_ratio);
    return s;
}

// BASELINE.json config 5, SURVEY.md 8(d): random_spheres_demo scaled to grid_side^2 spheres in
// ONE reference-built BVH.  grid_side = 1000 is the quoted configuration.  One deviation from
// SURVEY 8(d): the whole scene sits 0.1 lower (ground plane y = -0.1, sphere centres y = 0.1).
// The reference's Checker is the 3-D product sin(10x)sin(10y)sin(10z) (src/material.rs:252); on
// a plane at exactly y = 0 its sign is the sign of a rounding error, i.e. not a defined image.
SceneConfig stress_spheres(uint32_t grid_side) {
    SceneConfig s;
    auto& rng = thread_rng();
    const float k = (float)grid_side / 1000.0f;
    const float ext = 600.0f * k;
    auto checker = arc<Checker>(solid(0.1f, 0.1f, 0.1f), solid(0.9f, 0.9f, 0.9f));
    s.world.push_back(rect(Rect::XZRect(-ext, ext, -ext, ext, -0.1f, arc<Lambertian>(checker))));
    const int half = (int)grid_side / 2;
    for (int a = -half; a < (int)grid_side - half; ++a)
        for (int b = -half; b < (int)grid_side - half; ++b) {
            float choose_mat = rng.gen_f32();
            float cx = (float)a + 0.9f * rng.gen_f32();
            float cz = (float)b + 0.9f * rng.gen_f32();
            s.world.push_back(arc<Sphere>(Vec3(cx, 0.1f, cz), 0.2f, random_small_sphere_material(choose_mat)));
        }
    auto light_shape = rect(Rect::XZRect(-ext, ext, -ext, ext, 80.0f * k,
                                         arc<DiffuseLight>(arc<SolidColor>(Vec3(1.0f, 0.77f, 0.56f) * 2.0f))));
    s.world.push_back(flip(light_shape));
    s.lights.push_back(light_shape);
    s.aspect_ratio = 16.0f / 9.0f;
    s.cam_iter = fixed(Vec3(0, 40.0f * k, 260.0f * k), Vec3(0, 0, 0), 40.0f, s.aspect_ratio);
    return s;
}

} // namespace vecchio
