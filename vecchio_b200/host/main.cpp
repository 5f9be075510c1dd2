// main.cpp -- the caller of the path: the reference's main() (src/main.rs:155-221) with the sample loop
// (main.rs:181-198) replaced by the C ABI.  Scene generation, `BVHNode::new`, the camera iterator, the frame
// loop and the P3 writer stay on the host; the scene is uploaded once and stays resident while the iterator
// turns the camera (RotatingCamera, src/scene.rs:48-91).  What the reference fixes at compile time
// (the scene number of main.rs:159-167, `width`, SAMPLES_PER_PIXEL, MAX_DEPTH) is a command-line option
// here, with the reference's values as defaults.
//
// Several GPUs in ONE process (--gpus N): vk_multi_* of the C ABI.  GPU k renders the global samples
// [k*spp/N, (k+1)*spp/N) of every pixel into its own integer accumulators and GPU 0 adds its peers' accumulators
// to its own by reading them over NVLink (SURVEY 8e; the torch.distributed launch of bench.py does the same sum
// with one NCCL reduce) -- the frame is bit-identical to the one-GPU frame.  There is no CPU render path: without
// a device vk_create fails and so does this program.
#include "../../include/vecchio_gpu.h"
#include "../../include/vecchio_host.h"

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <future>
#include <string>
#include <thread>
#include <vector>

namespace {

const char* const kSceneByNumber[] = {"bowser_demo", "cornell_box", "final_scene", "random_spheres_demo",
                                      "perlin_demo", "balls_demo"}; // src/main.rs:160-165

struct Options {
    std::string scene = "cornell_box"; // `match 1` (main.rs:159)
    uint32_t scene_param = 0;
    uint32_t width = 900;   // main.rs:171
    uint32_t spp = 1000;    // SAMPLES_PER_PIXEL (main.rs:27)
    uint32_t max_depth = 100; // MAX_DEPTH (main.rs:28)
    uint32_t frames = 0;    // 0 = until cam_iter is exhausted (main.rs:176)
    uint32_t first_frame = 0;
    uint64_t seed = 1, scene_seed = 1;
    std::vector<int> devices{0};
    std::string out_dir, assets_dir = "assets";
    uint32_t variant = VK_VARIANT_AUTO, flags = 0;
    uint32_t batch = 1; // cameras per launch (vk_render_frames_rgb8); 1 = one vk_render_rgb8 per camera
    float adaptive = -1.0f; // >= 0: vk_render_adaptive_rgb8 with this max_error, --spp the cap
    uint32_t pass_spp = 0;  // its samples per pass (0 = not given: 64)
    bool quiet = false;
};

void usage(FILE* f) {
    std::fputs(
        "usage: vecchio_gpu_render [options]\n"
        "  --scene N|NAME     0 bowser_demo, 1 cornell_box (default), 2 final_scene, 3 random_spheres_demo,\n"
        "                     4 perlin_demo, 5 balls_demo (src/main.rs:159-167); by name also cornell_smoke,\n"
        "                     stress_spheres, api_surface_demo, random_spheres_cover, book1_cover,\n"
        "                     furnace_demo\n"
        "  --param K          scene parameter (stress_spheres: grid side)\n"
        "  --width W          image width, height = (W / aspect_ratio) as usize (default 900)\n"
        "  --spp S            SAMPLES_PER_PIXEL (default 1000)\n"
        "  --depth D          MAX_DEPTH (default 100)\n"
        "  --frames K         stop after K frames (default: the whole camera iterator)\n"
        "  --first-frame F    skip the first F cameras (file numbering is kept)\n"
        "  --seed S           Philox key of the render (default 1); frame f uses S + f\n"
        "  --batch K          render up to K cameras per launch (default 1).  Same files, byte for byte, with\n"
        "                     --strict or an explicit --variant; with auto in the render build a batch may run a\n"
        "                     faster kernel than one frame does, whose rounding differs (DESIGN.md section 7)\n"
        "  --adaptive E       adaptive sampling (vk_render_adaptive_rgb8): a pixel stops when half the width of\n"
        "                     sqrt(mean +- standard error) is <= E 8-bit steps in every channel, or at --spp samples\n"
        "                     (the cap).  E = 0 writes the same files as without --adaptive.  The stopping rule\n"
        "                     makes the estimate slightly biased.  One device, --batch 1 (DESIGN.md section 7)\n"
        "  --pass-spp M       samples per adaptive pass (default 64)\n"
        "  --scene-seed S     host RNG seed for scene generation and BVH axis choices (default 1)\n"
        "  --gpus N           render each frame on devices 0..N-1 (spp split N ways)\n"
        "  --devices a,b,..   explicit device list\n"
        "  --out-dir DIR      where output_NNNN.ppm go (default: current directory)\n"
        "  --assets DIR       directory of earthmap.png etc. (default: assets)\n"
        "  --variant V        auto | megakernel | wavefront | staged | warpq | stepq\n"
        "  --strict           reference operation order (no FMA contraction)\n"
        "  --legacy           book-1/2 integrator: Material::scatter, no light sampling\n"
        "  --sky              sky-gradient background (with --legacy)\n"
        "  --quiet            no per-frame line on stderr\n",
        f);
}

bool parse_u32(const char* s, uint32_t& out) {
    char* end = nullptr;
    unsigned long v = std::strtoul(s, &end, 10);
    if (!s[0] || *end || v > 0xFFFFFFFFul) return false;
    out = (uint32_t)v;
    return true;
}

// returns 0 = run, 1 = exit successfully (help), 2 = bad usage
int parse(int argc, char** argv, Options& o) {
    for (int i = 1; i < argc; i++) {
        std::string a = argv[i];
        auto need = [&](const char*& v) {
            if (i + 1 >= argc) {
                std::fprintf(stderr, "vecchio_gpu_render: %s needs a value\n", a.c_str());
                return false;
            }
            v = argv[++i];
            return true;
        };
        const char* v = nullptr;
        uint32_t u = 0;
        if (a == "--help" || a == "-h") {
            usage(stdout);
            return 1;
        } else if (a == "--scene") {
            if (!need(v)) return 2;
            if (parse_u32(v, u)) {
                if (u >= sizeof(kSceneByNumber) / sizeof(kSceneByNumber[0])) {
                    std::fprintf(stderr, "Not a valid scene\n"); // panic!("Not a valid scene") main.rs:166
                    return 2;
                }
                o.scene = kSceneByNumber[u];
            } else
                o.scene = v;
        } else if (a == "--param") {
            if (!need(v) || !parse_u32(v, o.scene_param)) return 2;
        } else if (a == "--width") {
            if (!need(v) || !parse_u32(v, o.width)) return 2;
        } else if (a == "--spp") {
            if (!need(v) || !parse_u32(v, o.spp)) return 2;
        } else if (a == "--depth") {
            if (!need(v) || !parse_u32(v, o.max_depth)) return 2;
        } else if (a == "--frames") {
            if (!need(v) || !parse_u32(v, o.frames)) return 2;
        } else if (a == "--batch") {
            if (!need(v) || !parse_u32(v, o.batch) || o.batch == 0) return 2;
        } else if (a == "--adaptive") {
            if (!need(v)) return 2;
            char* end = nullptr;
            const float e = std::strtof(v, &end);
            if (!v[0] || *end || !std::isfinite(e) || e < 0.0f) {
                std::fprintf(stderr, "vecchio_gpu_render: --adaptive needs a finite value >= 0\n");
                return 2;
            }
            o.adaptive = e;
        } else if (a == "--pass-spp") {
            if (!need(v) || !parse_u32(v, o.pass_spp) || o.pass_spp == 0) {
                std::fprintf(stderr, "vecchio_gpu_render: --pass-spp needs an integer >= 1\n");
                return 2;
            }
        } else if (a == "--first-frame") {
            if (!need(v) || !parse_u32(v, o.first_frame)) return 2;
        } else if (a == "--seed") {
            if (!need(v)) return 2;
            o.seed = std::strtoull(v, nullptr, 10);
        } else if (a == "--scene-seed") {
            if (!need(v)) return 2;
            o.scene_seed = std::strtoull(v, nullptr, 10);
        } else if (a == "--gpus") {
            if (!need(v) || !parse_u32(v, u) || u == 0 || u > 64) return 2;
            o.devices.clear();
            for (uint32_t d = 0; d < u; d++) o.devices.push_back((int)d);
        } else if (a == "--devices") {
            if (!need(v)) return 2;
            o.devices.clear();
            std::string list = v;
            size_t pos = 0;
            while (pos <= list.size()) {
                size_t comma = list.find(',', pos);
                if (comma == std::string::npos) comma = list.size();
                if (!parse_u32(list.substr(pos, comma - pos).c_str(), u)) return 2;
                o.devices.push_back((int)u);
                pos = comma + 1;
            }
            if (o.devices.empty()) return 2;
        } else if (a == "--out-dir") {
            if (!need(v)) return 2;
            o.out_dir = v;
        } else if (a == "--assets") {
            if (!need(v)) return 2;
            o.assets_dir = v;
        } else if (a == "--variant") {
            if (!need(v)) return 2;
            std::string s = v;
            if (s == "auto") o.variant = VK_VARIANT_AUTO;
            else if (s == "megakernel") o.variant = VK_VARIANT_MEGAKERNEL;
            else if (s == "wavefront") o.variant = VK_VARIANT_WAVEFRONT;
            else if (s == "staged") o.variant = VK_VARIANT_STAGED;
            else if (s == "warpq") o.variant = VK_VARIANT_WARPQ;
            else if (s == "stepq") o.variant = VK_VARIANT_STEPQ;
            else return 2;
        } else if (a == "--strict") {
            o.flags |= VK_FLAG_STRICT_MATH;
        } else if (a == "--legacy") {
            o.flags |= VK_FLAG_LEGACY_SCATTER;
        } else if (a == "--sky") {
            o.flags |= VK_FLAG_SKY_BACKGROUND;
        } else if (a == "--quiet") {
            o.quiet = true;
        } else {
            std::fprintf(stderr, "vecchio_gpu_render: unknown option %s\n", a.c_str());
            return 2;
        }
    }
    if (o.width < 2 || o.spp == 0 || o.spp < o.devices.size()) {
        std::fprintf(stderr, "vecchio_gpu_render: need width >= 2 and spp >= number of devices\n");
        return 2;
    }
    if (o.pass_spp && o.adaptive < 0.0f) {
        std::fprintf(stderr, "vecchio_gpu_render: --pass-spp needs --adaptive\n");
        return 2;
    }
    if (o.adaptive >= 0.0f && (o.batch > 1 || o.devices.size() > 1)) {
        std::fprintf(stderr, "vecchio_gpu_render: --adaptive renders one frame per call on one device (no --batch > 1, no --gpus > 1)\n");
        return 2;
    }
    if (!o.pass_spp) o.pass_spp = 64;
    return 0;
}

// one device: vk_ctx; several: vk_multi (spp slices per device, the peers' accumulators added on device 0 over NVLink)
struct Gpus {
    vk_ctx* one = nullptr;
    vk_multi* many = nullptr;
    const char* error() const { return many ? vk_multi_last_error(many) : vk_last_error(one); }
};

void destroy_all(Gpus& g, vkh_scene* scene) {
    if (g.one) vk_destroy(g.one);
    if (g.many) vk_multi_destroy(g.many);
    g.one = nullptr;
    g.many = nullptr;
    if (scene) vkh_scene_free(scene);
}

// --batch K > 1: the frame loop with up to K cameras of cam_iter per vk_render_frames_rgb8 (or
// vk_multi_render_frames_rgb8) call.  Frame f of a batch is file number n0 + f with seed + n0 + f -- the numbers and seeds
// of the one-camera loop, so the files are the same byte for byte whenever the batch runs the kernel a single frame runs:
// always with --strict (every kernel computes the reference's operation sequence) or an explicit --variant; with AUTO in
// the render build a batch that crosses AUTO's path-count rule runs another kernel, which rounds differently.  The P3 files of a batch are written by a helper
// thread while the next batch renders; one "Wrote frame" line per file.  Returns the exit code.
int render_batched(const Options& opt, Gpus& gpus, vkh_scene* scene, uint32_t width, uint32_t height) {
    const uint32_t world = (uint32_t)opt.devices.size();
    const size_t n_bytes = (size_t)width * height * 3;
    std::vector<uint8_t> rgb8_buf[2] = {std::vector<uint8_t>(n_bytes * opt.batch), std::vector<uint8_t>(n_bytes * opt.batch)};
    std::vector<vk_camera> cams;
    cams.reserve(opt.batch);
    struct Pending {
        std::future<std::string> done; // "" = written, else the writer's error message
        std::vector<std::string> filenames;
        std::chrono::steady_clock::time_point start;
        uint64_t rays = 0;
    } pending;
    auto finish_pending = [&]() -> bool {
        if (!pending.done.valid()) return true;
        std::string err = pending.done.get();
        if (!err.empty()) {
            std::fprintf(stderr, "vecchio_gpu_render: %s\n", err.c_str());
            return false;
        }
        if (!opt.quiet) { // the batch's time, shared evenly by its frames
            const double k = (double)pending.filenames.size();
            const double s = std::chrono::duration<double>(std::chrono::steady_clock::now() - pending.start).count() / k;
            for (const std::string& name : pending.filenames)
                std::fprintf(stderr, "Wrote frame %s in %.3fs (%.1f Mpaths/s, %.1f Mrays/s)\n", name.c_str(), s,
                             (double)width * height * opt.spp / s * 1e-6, (double)pending.rays / k / s * 1e-6);
        }
        return true;
    };
    uint32_t file_idx = 0, written = 0, n_batches = 0;
    bool cameras_left = true;
    while (cameras_left && !(opt.frames && written >= opt.frames)) {
        // the next up to K cameras of cam_iter (main.rs:176), after --first-frame, within --frames
        cams.clear();
        uint32_t first_idx = 0;
        while (cams.size() < opt.batch && !(opt.frames && written + cams.size() >= opt.frames)) {
            vk_camera cam;
            if (!vkh_scene_next_camera(scene, &cam)) {
                cameras_left = false;
                break;
            }
            if (file_idx < opt.first_frame) {
                file_idx++;
                continue;
            }
            if (cams.empty()) first_idx = file_idx;
            cams.push_back(cam);
            file_idx++;
        }
        if (cams.empty()) break;
        const uint32_t n = (uint32_t)cams.size();
        auto start = std::chrono::steady_clock::now();
        std::vector<uint8_t>& rgb8 = rgb8_buf[n_batches & 1];

        vk_render_params P{};
        P.width = width;
        P.height = height;
        P.spp = opt.spp;
        P.max_depth = opt.max_depth;
        P.seed = opt.seed + first_idx; // frame f of the batch: seed + first_idx + f
        P.variant = opt.variant;
        P.flags = opt.flags;
        vk_stats stats{};
        if ((world == 1 ? vk_render_frames_rgb8(gpus.one, cams.data(), n, &P, rgb8.data(), &stats)
                        : vk_multi_render_frames_rgb8(gpus.many, cams.data(), n, &P, rgb8.data(), &stats)) != VK_OK) {
            std::fprintf(stderr, "vecchio_gpu_render: %s\n", gpus.error());
            finish_pending();
            return 1;
        }
        // the previous batch's files are done before its buffer is reused by the batch after this one
        if (!finish_pending()) return 1;
        std::vector<std::string> names;
        for (uint32_t f = 0; f < n; f++) {
            char filename[4096];
            if (vkh_frame_filename(opt.out_dir.c_str(), first_idx + f, filename, sizeof filename) < 0) {
                std::fprintf(stderr, "vecchio_gpu_render: output path too long\n");
                return 1;
            }
            names.push_back(filename);
        }
        pending.filenames = names;
        pending.start = start;
        pending.rays = stats.rays;
        const uint8_t* data = rgb8.data();
        pending.done = std::async(std::launch::async, [data, width, height, n_bytes, names = std::move(names)]() -> std::string {
            for (size_t f = 0; f < names.size(); f++) // vkh_last_error is per thread: read it on the thread that failed
                if (vkh_write_ppm(names[f].c_str(), data + f * n_bytes, width, height) != VK_OK) return std::string(vkh_last_error());
            return std::string();
        });
        written += n;
        n_batches++;
    }
    return finish_pending() ? 0 : 1;
}

} // namespace

int main(int argc, char** argv) {
    Options opt;
    int pr = parse(argc, argv, opt);
    if (pr == 1) return 0;
    if (pr == 2) {
        usage(stderr);
        return 2;
    }

    // Camera and world (main.rs:156-169)
    std::fprintf(stderr, "Generating scene...\n");
    vkh_scene* scene = nullptr;
    if (vkh_scene_build(opt.scene.c_str(), opt.scene_seed, opt.assets_dir.c_str(), opt.scene_param, &scene) != VK_OK) {
        std::fprintf(stderr, "vecchio_gpu_render: %s\n", vkh_last_error());
        return 1;
    }
    const uint32_t width = opt.width;
    const uint32_t height = (uint32_t)((float)width / vkh_scene_aspect_ratio(scene)); // main.rs:172
    if (height < 2) {
        std::fprintf(stderr, "vecchio_gpu_render: image height %u is too small\n", height);
        vkh_scene_free(scene);
        return 2;
    }

    // the scene stays resident on every device for the whole frame loop
    Gpus gpus;
    const uint32_t world = (uint32_t)opt.devices.size();
    if (world == 1) {
        if (vk_create(opt.devices[0], &gpus.one) != VK_OK) {
            std::fprintf(stderr, "vecchio_gpu_render: device %d: %s\n", opt.devices[0], vk_last_error(nullptr));
            destroy_all(gpus, scene);
            return 1;
        }
    } else if (vk_multi_create(opt.devices.data(), (int)world, &gpus.many) != VK_OK) {
        std::fprintf(stderr, "vecchio_gpu_render: %s\n", vk_multi_last_error(nullptr));
        destroy_all(gpus, scene);
        return 1;
    }
    if ((world == 1 ? vk_scene_upload(gpus.one, vkh_scene_desc(scene)) : vk_multi_scene_upload(gpus.many, vkh_scene_desc(scene))) != VK_OK) {
        std::fprintf(stderr, "vecchio_gpu_render: %s\n", gpus.error());
        destroy_all(gpus, scene);
        return 1;
    }
    if (opt.batch > 1) {
        const int rc = render_batched(opt, gpus, scene, width, height);
        destroy_all(gpus, scene);
        return rc;
    }
    const size_t n_floats = (size_t)width * height * 3;
    // two output buffers: the P3 text of frame f is written by a helper thread while frame f+1 renders
    std::vector<uint8_t> rgb8_buf[2] = {std::vector<uint8_t>(n_floats), std::vector<uint8_t>(n_floats)};
    struct Pending {
        std::future<std::string> done; // "" = written, else the writer's error message
        std::string filename;
        std::chrono::steady_clock::time_point start;
        uint64_t rays = 0, paths = 0;
    } pending;
    auto finish_pending = [&]() -> bool {
        if (!pending.done.valid()) return true;
        std::string err = pending.done.get();
        if (!err.empty()) {
            std::fprintf(stderr, "vecchio_gpu_render: %s\n", err.c_str());
            return false;
        }
        if (!opt.quiet) {
            double s = std::chrono::duration<double>(std::chrono::steady_clock::now() - pending.start).count();
            std::fprintf(stderr, "Wrote frame %s in %.3fs (%.1f Mpaths/s, %.1f Mrays/s)\n", pending.filename.c_str(), s,
                         (double)pending.paths / s * 1e-6, (double)pending.rays / s * 1e-6);
        }
        return true;
    };
    uint32_t file_idx = 0, written = 0;
    vk_camera cam;
    while (vkh_scene_next_camera(scene, &cam)) { // for cam in config.cam_iter (main.rs:176)
        if (file_idx < opt.first_frame) {
            file_idx++;
            continue;
        }
        if (opt.frames && written >= opt.frames) break;
        auto start = std::chrono::steady_clock::now();
        std::vector<uint8_t>& rgb8 = rgb8_buf[written & 1];

        vk_render_params P{};
        P.width = width;
        P.height = height;
        P.spp = opt.spp;
        P.max_depth = opt.max_depth;
        P.seed = opt.seed + file_idx;
        P.variant = opt.variant;
        P.flags = opt.flags;

        // sample loop + Vec3::to_color on the device(s); a quarter of the bytes come back
        vk_stats stats{};
        const int rc = opt.adaptive >= 0.0f ? vk_render_adaptive_rgb8(gpus.one, &cam, &P, opt.pass_spp, opt.adaptive, rgb8.data(), nullptr, &stats)
                       : world == 1        ? vk_render_rgb8(gpus.one, &cam, &P, rgb8.data(), &stats)
                                           : vk_multi_render_rgb8(gpus.many, &cam, &P, rgb8.data(), &stats);
        if (rc != VK_OK) {
            std::fprintf(stderr, "vecchio_gpu_render: %s\n", gpus.error());
            destroy_all(gpus, scene);
            return 1;
        }
        const uint64_t rays = stats.rays;

        // Write output (main.rs:200-214), overlapped with the next frame's render.  At most one write is in
        // flight, so the other buffer is free by the time the next frame is converted into it.
        if (!finish_pending()) {
            destroy_all(gpus, scene);
            return 1;
        }
        char filename[4096];
        if (vkh_frame_filename(opt.out_dir.c_str(), file_idx, filename, sizeof filename) < 0) {
            std::fprintf(stderr, "vecchio_gpu_render: output path too long\n");
            destroy_all(gpus, scene);
            return 1;
        }
        pending.filename = filename;
        pending.start = start;
        pending.rays = rays;
        pending.paths = opt.adaptive >= 0.0f ? stats.paths : (uint64_t)width * height * opt.spp;
        const uint8_t* data = rgb8.data();
        pending.done = std::async(std::launch::async, [data, width, height, name = pending.filename]() -> std::string {
            // vkh_last_error is per thread: read it on the thread that failed
            return vkh_write_ppm(name.c_str(), data, width, height) == VK_OK ? std::string() : std::string(vkh_last_error());
        });
        file_idx++;
        written++;
    }
    const bool ok = finish_pending();
    destroy_all(gpus, scene);
    return ok ? 0 : 1;
}
