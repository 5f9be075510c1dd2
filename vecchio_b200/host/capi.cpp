// capi.cpp -- extern "C" view of the host front end (include/vecchio_host.h).
#include "../../include/vecchio_host.h"
#include "vecchio.hpp"
#include <array>
#include <cerrno>
#include <cmath>
#include <cstdio>
#include <cstring>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif

using namespace vecchio;

struct vkh_scene {
    std::unique_ptr<LoweredScene> scene;
    vk_scene_desc desc;
};

static thread_local std::string g_err;

extern "C" {

int vkh_scene_build(const char* name, uint64_t seed, const char* assets_dir, uint32_t param, vkh_scene** out) {
    if (!name || !out) {
        g_err = "vkh_scene_build: null argument";
        return VK_ERR_INVALID;
    }
    try {
        g_assets_dir = assets_dir ? assets_dir : "assets";
        seed_thread_rng(seed);
        std::string n(name);
        SceneConfig cfg;
        if (n == "balls_demo") cfg = balls_demo();
        else if (n == "random_spheres_demo") cfg = random_spheres_demo();
        else if (n == "random_spheres_cover") cfg = random_spheres_cover();
        else if (n == "api_surface_demo") cfg = api_surface_demo();
        else if (n == "book1_cover") cfg = book1_cover();
        else if (n == "furnace_demo") cfg = furnace_demo(param);
        else if (n == "perlin_demo") cfg = perlin_demo();
        else if (n == "bowser_demo") cfg = bowser_demo();
        else if (n == "cornell_box") cfg = cornell_box();
        else if (n == "final_scene") cfg = final_scene();
        else if (n == "cornell_smoke") cfg = cornell_smoke();
        else if (n == "stress_spheres") cfg = stress_spheres(param ? param : 1000);
        else {
            g_err = "Not a valid scene: " + n; // panic!("Not a valid scene") src/main.rs:166
            return VK_ERR_INVALID;
        }
        auto s = new vkh_scene;
        s->scene = lower_scene(std::move(cfg));
        s->desc = s->scene->low.desc();
        *out = s;
        return VK_OK;
    } catch (const LowerError& e) {
        g_err = e.what();
        return VK_ERR_UNSUPPORTED;
    } catch (const std::exception& e) {
        g_err = e.what();
        return VK_ERR_INVALID;
    }
}

void vkh_scene_free(vkh_scene* s) { delete s; }
const vk_scene_desc* vkh_scene_desc(const vkh_scene* s) { return s ? &s->desc : nullptr; }
float vkh_scene_aspect_ratio(const vkh_scene* s) { return s ? s->scene->aspect_ratio : 0.0f; }

int vkh_scene_next_camera(vkh_scene* s, vk_camera* out) {
    if (!s || !out || !s->scene->cam_iter) return 0;
    auto c = s->scene->cam_iter->next();
    if (!c) return 0;
    *out = c->lower();
    return 1;
}

void vkh_camera_new(const float lookfrom[3], const float lookat[3], const float vup[3], float vfov,
                    float aspect_ratio, float aperture, float focus_dist, float time0, float time1,
                    vk_camera* out) {
    Camera c = Camera::make(Vec3(lookfrom[0], lookfrom[1], lookfrom[2]), Vec3(lookat[0], lookat[1], lookat[2]),
                            Vec3(vup[0], vup[1], vup[2]), vfov, aspect_ratio, aperture, focus_dist, time0, time1);
    *out = c.lower();
}

long vkh_decode_png(const char* path, uint8_t* buf, size_t buf_len, uint32_t* width, uint32_t* height) {
    try {
        ImageTexture t(path);
        if (width) *width = (uint32_t)t.width;
        if (height) *height = (uint32_t)t.height;
        if (buf) {
            if (buf_len < t.buf.size()) {
                g_err = "vkh_decode_png: buffer too small";
                return -1;
            }
            std::memcpy(buf, t.buf.data(), t.buf.size());
        }
        return (long)t.buf.size();
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}

// Vec3::to_color (src/vec3.rs:54-61) for one channel.  Vec3::clamp (src/vec3.rs:44-52) is two `<`/`>` tests,
// so NaN falls through it and `NaN as u32` is 0.  Written without branches so the row loop vectorises:
// the two selects mirror the two tests, and the final select on v == v is the NaN -> 0 of the cast.
static inline uint8_t to_color1(float c) {
    float x = std::sqrt(c);
    x = x < 0.0f ? 0.0f : x;
    x = x > 0.999f ? 0.999f : x;
    float v = 256.0f * x;
    v = v == v ? v : 0.0f;
    return (uint8_t)(int)v; // 0 <= v < 256
}

void vkh_frame_to_rgb8(const float* frame, uint32_t width, uint32_t height, uint8_t* out_rgb8) {
    if (!frame || !out_rgb8) return;
    const size_t row_len = (size_t)width * 3;
    for (uint32_t row = 0; row < height; row++) { // file row `row` = image row height-1-row (main.rs:209)
        const float* src = frame + (size_t)(height - 1 - row) * row_len;
        uint8_t* dst = out_rgb8 + (size_t)row * row_len;
        size_t i = 0;
#if defined(__SSE2__)
        // 16 channels per step.  sqrtps is correctly rounded like sqrtf; maxps/minps return their SECOND operand
        // when the first is NaN, so max(x, 0) already turns NaN into the 0 that `NaN as u32` gives.
        const __m128 zero = _mm_setzero_ps(), top = _mm_set1_ps(0.999f), scale = _mm_set1_ps(256.0f);
        for (; i + 16 <= row_len; i += 16) {
            __m128i q[4];
            for (int k = 0; k < 4; k++) {
                __m128 x = _mm_sqrt_ps(_mm_loadu_ps(src + i + 4 * k));
                x = _mm_min_ps(_mm_max_ps(x, zero), top);
                q[k] = _mm_cvttps_epi32(_mm_mul_ps(scale, x));
            }
            __m128i lo = _mm_packs_epi32(q[0], q[1]), hi = _mm_packs_epi32(q[2], q[3]);
            _mm_storeu_si128((__m128i*)(dst + i), _mm_packus_epi16(lo, hi));
        }
#endif
        for (; i < row_len; i++) dst[i] = to_color1(src[i]);
    }
}

int vkh_write_ppm(const char* path, const uint8_t* rgb8, uint32_t width, uint32_t height) {
    if (!path || !rgb8) {
        g_err = "vkh_write_ppm: null argument";
        return VK_ERR_INVALID;
    }
    FILE* f = std::fopen(path, "wb");
    if (!f) {
        g_err = std::string("vkh_write_ppm: cannot create ") + path + ": " + std::strerror(errno);
        return VK_ERR_INVALID;
    }
    std::setvbuf(f, nullptr, _IONBF, 0); // the text is assembled in 1 MiB blocks below
    // the decimal text of 0..255 followed by a blank, and its length; a pixel line is at most
    // "255 255 255\n" = 12 bytes, written as three 4-byte stores of which the cursor keeps 2..4
    struct Dec {
        char text[4];
        uint32_t len;
    };
    static const std::array<Dec, 256> dec = [] {
        std::array<Dec, 256> t{};
        for (int v = 0; v < 256; v++) {
            char tmp[8];
            int n = std::snprintf(tmp, sizeof tmp, "%d ", v);
            std::memcpy(t[v].text, tmp, 4);
            t[v].len = (uint32_t)n;
        }
        return t;
    }();
    const size_t kBlock = 1u << 20;
    std::vector<char> buf(kBlock + 16);
    char* cur = buf.data();
    cur += std::snprintf(cur, 64, "P3\n%u %u\n255\n", width, height);
    bool ok = true;
    const size_t n_pixels = (size_t)width * height;
    const uint8_t* px = rgb8;
    for (size_t i = 0; i < n_pixels && ok; i++, px += 3) {
        std::memcpy(cur, dec[px[0]].text, 4);
        cur += dec[px[0]].len;
        std::memcpy(cur, dec[px[1]].text, 4);
        cur += dec[px[1]].len;
        std::memcpy(cur, dec[px[2]].text, 4);
        cur += dec[px[2]].len;
        cur[-1] = '\n';
        if ((size_t)(cur - buf.data()) >= kBlock) {
            ok = std::fwrite(buf.data(), 1, (size_t)(cur - buf.data()), f) == (size_t)(cur - buf.data());
            cur = buf.data();
        }
    }
    if (ok && cur != buf.data()) ok = std::fwrite(buf.data(), 1, (size_t)(cur - buf.data()), f) == (size_t)(cur - buf.data());
    if (std::fclose(f) != 0) ok = false;
    if (!ok) {
        g_err = std::string("vkh_write_ppm: write failed on ") + path;
        return VK_ERR_INVALID;
    }
    return VK_OK;
}

int vkh_write_pfm(const char* path, const float* data, uint32_t width, uint32_t height, uint32_t channels) {
    if (!path || !data || (channels != 1 && channels != 3)) {
        g_err = "vkh_write_pfm: null argument or channels other than 1 and 3";
        return VK_ERR_INVALID;
    }
    FILE* f = std::fopen(path, "wb");
    if (!f) {
        g_err = std::string("vkh_write_pfm: cannot create ") + path + ": " + std::strerror(errno);
        return VK_ERR_INVALID;
    }
    bool ok = std::fprintf(f, "%s\n%u %u\n-1.0\n", channels == 3 ? "PF" : "Pf", width, height) > 0;
    // the floats as little-endian bytes whatever the host's byte order, one row at a time
    std::vector<unsigned char> row((size_t)width * channels * 4);
    for (uint32_t y = 0; ok && y < height; ++y) {
        const float* src = data + (size_t)y * width * channels;
        for (size_t i = 0; i < (size_t)width * channels; ++i) {
            uint32_t b;
            std::memcpy(&b, src + i, 4);
            for (int k = 0; k < 4; ++k) row[4 * i + k] = (unsigned char)(b >> (8 * k));
        }
        ok = std::fwrite(row.data(), 1, row.size(), f) == row.size();
    }
    if (std::fclose(f) != 0 || !ok) {
        g_err = std::string("vkh_write_pfm: write failed on ") + path;
        return VK_ERR_INVALID;
    }
    return VK_OK;
}

int vkh_frame_filename(const char* dir, uint32_t file_idx, char* buf, size_t buf_len) {
    if (!buf) return -1;
    const bool has_dir = dir && dir[0];
    const bool slash = has_dir && dir[std::strlen(dir) - 1] == '/';
    int n = std::snprintf(buf, buf_len, "%s%soutput_%04u.ppm", has_dir ? dir : "", has_dir && !slash ? "/" : "", file_idx);
    return n < 0 || (size_t)n >= buf_len ? -1 : n;
}

const char* vkh_last_error(void) { return g_err.c_str(); }

} // extern "C"
