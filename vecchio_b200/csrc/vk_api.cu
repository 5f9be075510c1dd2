// vk_api.cu -- the C ABI of include/vecchio_gpu.h: context, scene validation + upload (with the
// GPU-side re-layout), render orchestration, the parity hook and the roofline microbenchmarks.
// No CPU fallback anywhere: every entry point either runs CUDA kernels or returns an error.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <thread>
#include <vector>

#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "vk_internal.h"
#include "vk_relayout.h"

using namespace vkhost;

struct vk_ctx {
    int device = 0;
    int sm_count = 0;
    int clock_khz = 0;
    char name[128] = {0};
    cudaStream_t stream = nullptr;     // stream all work is enqueued on
    cudaStream_t own_stream = nullptr; // the one created by vk_create
    uint64_t launches = 0;             // kernels launched since the last stats read
    uint64_t paths = 0;                // samples started since the last stats read
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
    std::string err;
    std::vector<void*> scene_allocs;
    // Scene arena: one device block the arrays of an upload are carved from, sized by the previous upload (a caller that
    // uploads per frame -- bench.py's e2e step -- pays ~20 cudaMalloc / cudaFree pairs per upload without it); arrays that
    // do not fit fall back to their own allocation (scene_allocs) and the block grows before the next upload.
    char* arena = nullptr;
    size_t arena_cap = 0, arena_used = 0, arena_need = 0;
    cudaEvent_t ev_chunk[4] = {nullptr, nullptr, nullptr, nullptr}; // readout: D2H in chunks, copy-out of one while the next arrives
    DScene scene{};
    FlatProgram flat{}; // flat.n == 0: scene too large, BVH traversal
    bool has_scene = false;
    uint32_t n_nodes = 0; // BVH nodes of the uploaded scene
    uint32_t n_materials = 0, n_textures = 0, n_media = 0;
    size_t wnodes_bytes = 0;                    // size of the 4-wide node array (the L2 access-policy window covers it)
    size_t l2_persist_max = 0, l2_window_max = 0; // device limits for persisting L2 lines / the policy window
    bool has_specdiffuse = false;
    bool simple_scene = false; // only what the VK_SIMPLE build of the staged kernel keeps (see vk_device.cuh)
    bool one_rect_light = false; // the light list is exactly one unflipped Rect: the VK_LIGHT0 builds apply
    uint32_t flat_shape = VKF_SHAPE_NONE; // the flat program's shape, if the trimmed warp-queue kernel is compiled for it
    unsigned long long* debug = nullptr;    // per-CTA diagnostics of the staged kernel (VK_DEBUG_CTAS x 4 words)
    unsigned long long* counters = nullptr; // [0] rays [1] dropped [2] work head
    float* partial = nullptr;               // accumulators: W*H*3 x u64 fixed-point sums | W*H*3 x double sums of squares
    size_t partial_floats = 0;
    float* sq_stack = nullptr; // step-queue kernel: overflow of the traversal stacks (allocated on first use)
    size_t sq_stack_floats = 0;
    uint32_t stack_need = 0, levels_sub = 0; // of the uploaded scene (vk_scene_info)
    float* frame = nullptr; // device staging of a render call's results (Staging)
    size_t frame_floats = 0;
    float* pinned = nullptr; // pinned host staging of the results' copy back (Staging), and of the adaptive pass loop's counts
    size_t pinned_floats = 0;
    DCamera* cams = nullptr; // vk_render_frames: the batch's cameras on the device (FrameArgs::cams)
    size_t cams_cap = 0;
    std::vector<DCamera> cams_host;
    vk_adaptive_session* oneshot = nullptr; // vk_render_adaptive*: the session each call begins, refines once and reads
    uint64_t scene_gen = 0;                 // scene uploads so far: a session refines only on the scene it began with
    // wavefront variant: the slot pool (allocated on first use) and a pinned word block for the
    // host's termination checks
    WfState wf{};
    void* wf_block = nullptr;
    uint32_t* wf_host_counts = nullptr;
};

static thread_local std::string g_create_err;
extern "C" {
static void adaptive_free(vk_adaptive_session* s); // (defined with the sessions, in the C ABI's block)
}

static int fail(vk_ctx* c, int code, const std::string& msg) {
    if (c) c->err = msg;
    else g_create_err = msg;
    return code;
}
#define CU(ctx, call)                                                                                                  \
    do {                                                                                                               \
        cudaError_t e_ = (call);                                                                                       \
        if (e_ != cudaSuccess)                                                                                         \
            return fail(ctx, e_ == cudaErrorMemoryAllocation ? VK_ERR_OOM : VK_ERR_CUDA,                               \
                        std::string(#call) + ": " + cudaGetErrorString(e_));                                           \
    } while (0)

// ------------------------------------------------------------------------------------------------
// small kernels that do not depend on the math mode
// ------------------------------------------------------------------------------------------------
// fixed-point accumulators -> fp32 per-pixel sums (the buffers the NCCL reduce combines)
__global__ void k_acc_to_sum(const unsigned long long* __restrict__ acc, const double* __restrict__ accsq, size_t n,
                             float* __restrict__ sum, float* __restrict__ sumsq) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    sum[i] = (float)((double)(long long)acc[i] * VK_ACC_INV_SCALE);
    if (sumsq) sumsq[i] = (float)accsq[i];
}
// Where the readout kernels take a pixel's mean from (k_finalize, k_to_color).  SumsOverSpp: float sums (k_acc_to_sum's or
// k_reduce_peers') over a constant spp, c /= SAMPLES_PER_PIXEL as f32 (src/main.rs:196).  AccOverCount: an adaptive state's
// fixed-point sums over each pixel's own count; it forms k_acc_to_sum's float sum, (float)((double)(long long)acc *
// VK_ACC_INV_SCALE), in a register and divides it by the float count as SumsOverSpp does, so a pixel that stopped at n
// samples reads out as vk_render(spp = n) does, bit for bit.
struct SumsOverSpp {
    static constexpr bool counted = false;
    const float* __restrict__ sum;
    float spp;
    __device__ float mean(size_t j) const { return sum[j] / spp; }
};
struct AccOverCount {
    static constexpr bool counted = true;
    const unsigned long long* __restrict__ acc;
    const uint32_t* __restrict__ nspp;
    __device__ float mean(size_t j) const { return (float)((double)(long long)acc[j] * VK_ACC_INV_SCALE) / (float)nspp[j / 3]; }
};
// The element of n_frames contiguous planes, in the accumulators' order (each frame's rows bottom-up), that element i of the
// same planes top-down holds (the order of an rgb8 image and of the PPM, src/main.rs:209); a row is width * per elements.
__device__ __forceinline__ size_t flip_rows(size_t i, uint32_t width, uint32_t height, uint32_t per) {
    const size_t row_len = (size_t)width * per, frame = row_len * height, f = i / frame, k = i - f * frame, row = k / row_len;
    return f * frame + (height - 1 - row) * row_len + (k - row * row_len);
}
template <class Src> __global__ void k_finalize(Src src, float* __restrict__ rgb, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) rgb[i] = src.mean(i);
}
// Vec3::to_color (src/vec3.rs:54-61) of the means of n_frames frames, each frame top-down on its own; spp_out (AccOverCount,
// nullable): the counts in the image's order
template <class Src>
__global__ void k_to_color(Src src, uint8_t* __restrict__ out, uint32_t* __restrict__ spp_out, uint32_t width, uint32_t height, uint32_t n_frames) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)width * height * 3 * n_frames) return;
    const size_t j = flip_rows(i, width, height, 3);
    float v = sqrtf(src.mean(j));
    v = v < 0.0f ? 0.0f : (v > 0.999f ? 0.999f : v); // Vec3::clamp keeps NaN
    out[i] = (uint8_t)__float2uint_rz(256.0f * v);   // `as u32`: NaN -> 0
    if constexpr (Src::counted)
        if (spp_out && i % 3 == 0) spp_out[i / 3] = src.nspp[j / 3];
}
// ---- adaptive sampling (vk_render_adaptive) ----
// The pixels shard `shard` of n_shards owns (include/vecchio_gpu.h, vk_adaptive_begin_shard): pixel g belongs to shard
// (g / VK_SHARD_RUN) mod n_shards.  A fresh refine's pass-0 list: the n_owned owned pixels of n_pix, ascending (entry i
// lies in the shard's run i / VK_SHARD_RUN); with one shard, every pixel.
__device__ __forceinline__ bool shard_owns(uint32_t p, uint32_t shard, uint32_t n_shards) {
    return (p / VK_SHARD_RUN) % n_shards == shard;
}
__global__ void k_shard_list(uint32_t* list, uint32_t n_owned, uint32_t shard, uint32_t n_shards) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_owned) list[i] = ((i / VK_SHARD_RUN) * n_shards + shard) * VK_SHARD_RUN + i % VK_SHARD_RUN;
}
// The largest channel error e of pixel p after n >= 2 samples (include/vecchio_gpu.h states it), from the integer sums
// alone, so that it does not depend on the order the samples arrived in.  Every operation is IEEE double, rounded to
// nearest (this file is built without -prec-div / -prec-sqrt = false), and q - m^2 is written as the one fused
// multiply-add it is: left to the compiler, each inlined copy could be contracted or not, and the one-shot kernel
// (k_adaptive_select) and a refine's (k_adaptive_levels) could then decide differently within an ulp of max_error.
// tests/adaptive_model.py restates the sequence on the host, bit for bit.
__device__ __forceinline__ double adaptive_error(const unsigned long long* __restrict__ acc, const unsigned long long* __restrict__ sq,
                                                 uint32_t p, uint32_t n) {
    double e = 0.0;
    for (uint32_t ch = 0; ch < 3u; ++ch) {
        const double m = (double)(long long)acc[3u * p + ch] * VK_ACC_INV_SCALE / n;
        const double q = (double)sq[3u * p + ch] * VK_SQ_INV_SCALE / n;
        const double se = sqrt(fmax(fma(-m, m, q), 0.0) / (double)(n - 1u));
        e = fmax(e, 128.0 * (sqrt(fmax(m + se, 0.0)) - sqrt(fmax(m - se, 0.0))));
    }
    return e;
}
// The stopping rule, the one place it is written: a pixel at n samples stops at the cap spp, or once n >= min_spp, n > 1
// (one sample has no standard error) and e <= max_error; max_error == 0 never stops early.
__device__ __forceinline__ bool adaptive_stop(const unsigned long long* __restrict__ acc, const unsigned long long* __restrict__ sq,
                                              uint32_t p, uint32_t n, uint32_t spp, uint32_t min_spp, float max_error) {
    bool stop = n >= spp;
    if (!stop && max_error > 0.0f && n > 1u && n >= min_spp) stop = adaptive_error(acc, sq, p, n) <= (double)max_error;
    return stop;
}
// The rule for every listed pixel after a pass that brought it to n_done samples: records n_done as its count,
// keep[i] = 1 when it renders on.
__global__ void k_adaptive_select(const uint32_t* __restrict__ list, uint32_t n, const unsigned long long* __restrict__ acc,
                                  const unsigned long long* __restrict__ sq, uint32_t n_done, uint32_t spp, uint32_t min_spp,
                                  float max_error, uint32_t* __restrict__ nspp, uint8_t* __restrict__ keep) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t p = list[i];
    nspp[p] = n_done;
    keep[i] = adaptive_stop(acc, sq, p, n_done, spp, min_spp, max_error) ? 0u : 1u;
}
// A refine of a session that already holds samples: the rule of the new target for every pixel below its cap.  level[p] =
// n_p / pass_spp + 1 for a pixel that renders on (its count is on the pass grid, see vk_adaptive_refine), 0 otherwise;
// n_level[l] counts the pixels that render on from level l (one atomic per warp and level).  A shard's pixels it does not
// own stay at level 0: they are never listed.
__global__ void k_adaptive_levels(const unsigned long long* __restrict__ acc, const unsigned long long* __restrict__ sq,
                                  const uint32_t* __restrict__ nspp, uint32_t n_pix, uint32_t spp, uint32_t min_spp, float max_error,
                                  uint32_t pass_spp, uint32_t shard, uint32_t n_shards, uint32_t* __restrict__ level,
                                  uint32_t* __restrict__ n_level) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t lv = 0;
    if (i < n_pix) {
        const uint32_t n = nspp[i];
        if (shard_owns(i, shard, n_shards) && !adaptive_stop(acc, sq, i, n, spp, min_spp, max_error)) lv = n / pass_spp + 1u;
        level[i] = lv;
    }
    const unsigned peers = __match_any_sync(0xFFFFFFFFu, lv);
    if (lv && (uint32_t)(__ffs(peers) - 1) == (threadIdx.x & 31u)) atomicAdd(&n_level[lv - 1u], (uint32_t)__popc(peers));
}
// The error map of a session: e per pixel as the rule sees it, +inf below two samples; top_down: each frame's rows
// top-down (the order of an rgb8 image), otherwise the accumulators' order
__global__ void k_adaptive_error_map(const unsigned long long* __restrict__ acc, const unsigned long long* __restrict__ sq,
                                     const uint32_t* __restrict__ nspp, float* __restrict__ out, uint32_t width, uint32_t height,
                                     uint32_t n_frames, bool top_down) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)width * height * n_frames) return;
    const size_t p = top_down ? flip_rows(i, width, height, 1) : i;
    const uint32_t n = nspp[p];
    out[i] = n < 2u ? __int_as_float(0x7F800000) : (float)adaptive_error(acc, sq, (uint32_t)p, n);
}
// FP32 peak: 8 independent FFMA chains per thread, no memory traffic
__global__ void k_ffma_peak(float* out, int iters) {
    float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f, a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f,
          a7 = a0 + 7.f;
    const float m = 0.999f, b = 1e-3f;
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            a0 = fmaf(a0, m, b); a1 = fmaf(a1, m, b); a2 = fmaf(a2, m, b); a3 = fmaf(a3, m, b);
            a4 = fmaf(a4, m, b); a5 = fmaf(a5, m, b); a6 = fmaf(a6, m, b); a7 = fmaf(a7, m, b);
        }
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}
// L2 bandwidth: every block streams the same L2-resident buffer with 128-bit loads
__global__ void k_l2_read(const float4* __restrict__ buf, size_t n_vec, int reps, float* out) {
    float acc = 0.f;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (int r = 0; r < reps; ++r)
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += stride) {
            const float4 v = __ldcg(&buf[i]);
            acc += v.x + v.y + v.z + v.w;
        }
    if (acc == 123.456f) out[0] = acc;
}

// (scene validation and layout planning: vk_relayout.h)
namespace {
template <class T> int upload(vk_ctx* c, const T* src, size_t n, const T** dst) {
    *dst = nullptr;
    if (n == 0) n = 1; // keep pointers valid
    void* p = nullptr;
    const size_t bytes = (n * sizeof(T) + 255) & ~(size_t)255;
    c->arena_need += bytes;
    if (c->arena && c->arena_used + bytes <= c->arena_cap) {
        p = c->arena + c->arena_used;
        c->arena_used += bytes;
    } else {
        CU(c, cudaMalloc(&p, n * sizeof(T)));
        c->scene_allocs.push_back(p);
    }
    if (src) CU(c, cudaMemcpyAsync(p, src, n * sizeof(T), cudaMemcpyHostToDevice, c->stream));
    *dst = (const T*)p;
    return VK_OK;
}
void free_scene(vk_ctx* c) {
    for (void* p : c->scene_allocs) cudaFree(p);
    c->scene_allocs.clear();
    c->arena_used = 0;
    c->has_scene = false;
}
int ensure(vk_ctx* c, float** buf, size_t* have, size_t want) {
    if (*have >= want) return VK_OK;
    if (*buf) cudaFree(*buf);
    *buf = nullptr;
    *have = 0;
    CU(c, cudaMalloc((void**)buf, want * sizeof(float)));
    *have = want;
    return VK_OK;
}
// the pinned counterpart: c->pinned, the host staging of the results, holds at least `floats` floats
static int ensure_pinned(vk_ctx* c, size_t floats) {
    if (c->pinned_floats >= floats) return VK_OK;
    if (c->pinned) cudaFreeHost(c->pinned);
    c->pinned = nullptr;
    c->pinned_floats = 0;
    CU(c, cudaMallocHost((void**)&c->pinned, floats * sizeof(float)));
    c->pinned_floats = floats;
    return VK_OK;
}
DCamera to_dcam(const vk_camera* k) {
    DCamera c;
    auto v3 = [](const float* p) { return make_float3(p[0], p[1], p[2]); };
    c.origin = v3(k->origin);
    c.lower_left_corner = v3(k->lower_left_corner);
    c.horizontal = v3(k->horizontal);
    c.vertical = v3(k->vertical);
    c.u = v3(k->u);
    c.v = v3(k->v);
    c.lens_radius = k->lens_radius;
    c.time0 = k->time0;
    c.time1 = k->time1;
    return c;
}
} // namespace

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

int vk_create(int device, vk_ctx** out) {
    if (!out) return fail(nullptr, VK_ERR_INVALID, "vk_create: null out pointer");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(nullptr, VK_ERR_NO_DEVICE, std::string("vk_create: no CUDA device (") + cudaGetErrorString(e) +
                                                   "); this library has no CPU fallback");
    if (device < 0 || device >= n) return fail(nullptr, VK_ERR_INVALID, "vk_create: device index out of range");
    vk_ctx* c = new vk_ctx;
    c->device = device;
#define CUC(call)                                                                                                      \
    do {                                                                                                               \
        cudaError_t e_ = (call);                                                                                       \
        if (e_ != cudaSuccess) {                                                                                       \
            g_create_err = std::string(#call) + ": " + cudaGetErrorString(e_);                                         \
            delete c;                                                                                                  \
            return VK_ERR_CUDA;                                                                                        \
        }                                                                                                              \
    } while (0)
    CUC(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUC(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        g_create_err = std::string("vk_create: device '") + prop.name + "' is sm_" + std::to_string(prop.major * 10 + prop.minor) +
                       "; this library is built for sm_100a only";
        delete c;
        return VK_ERR_NO_DEVICE;
    }
    c->sm_count = prop.multiProcessorCount;
    c->l2_persist_max = (size_t)prop.persistingL2CacheMaxSize;
    c->l2_window_max = (size_t)prop.accessPolicyMaxWindowSize;
    if (c->l2_persist_max) cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, c->l2_persist_max); // used by large BVHs only
    cudaGetLastError();
    c->clock_khz = prop.clockRate;
    std::snprintf(c->name, sizeof(c->name), "%.100s", prop.name);
    CUC(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
    c->stream = c->own_stream;
    CUC(cudaEventCreate(&c->ev0));
    CUC(cudaEventCreate(&c->ev1));
    CUC(cudaEventCreate(&c->ev2));
    CUC(cudaMalloc((void**)&c->counters, 8 * sizeof(unsigned long long)));
    CUC(cudaMemset(c->counters, 0, 8 * sizeof(unsigned long long)));
    CUC(cudaMalloc((void**)&c->debug, VK_DEBUG_CTAS * 4 * sizeof(unsigned long long)));
    CUC(cudaMemset(c->debug, 0, VK_DEBUG_CTAS * 4 * sizeof(unsigned long long)));
#undef CUC
    *out = c;
    return VK_OK;
}

void vk_destroy(vk_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    free_scene(c);
    if (c->arena) cudaFree(c->arena);
    for (cudaEvent_t e : c->ev_chunk)
        if (e) cudaEventDestroy(e);
    if (c->partial) cudaFree(c->partial);
    if (c->sq_stack) cudaFree(c->sq_stack);
    if (c->wf_block) cudaFree(c->wf_block);
    if (c->wf_host_counts) cudaFreeHost(c->wf_host_counts);
    if (c->frame) cudaFree(c->frame);
    if (c->pinned) cudaFreeHost(c->pinned);
    if (c->cams) cudaFree(c->cams);
    adaptive_free(c->oneshot);
    if (c->counters) cudaFree(c->counters);
    if (c->debug) cudaFree(c->debug);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->ev2) cudaEventDestroy(c->ev2);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
}

const char* vk_last_error(const vk_ctx* c) { return c ? c->err.c_str() : g_create_err.c_str(); }

int vk_device_info(vk_ctx* c, int* sm_count, int* clock_khz, char* name, size_t name_len) {
    if (!c) return VK_ERR_INVALID;
    if (sm_count) *sm_count = c->sm_count;
    if (clock_khz) *clock_khz = c->clock_khz;
    if (name && name_len) std::snprintf(name, name_len, "%s", c->name);
    return VK_OK;
}

int vk_scene_upload(vk_ctx* c, const vk_scene_desc* d) {
    if (!c) return VK_ERR_INVALID;
    if (!d) return fail(c, VK_ERR_INVALID, "vk_scene_upload: null scene");
    Validator v;
    v.d = d;
    if (!v.run()) return fail(c, v.code, "vk_scene_upload: " + v.err);
    CU(c, cudaSetDevice(c->device));
    free_scene(c);
    ++c->scene_gen;
    if (c->arena_need > c->arena_cap) { // the previous upload did not fit: grow (cudaFree waits for the work that reads the old block)
        if (c->arena) cudaFree(c->arena);
        c->arena = nullptr;
        c->arena_cap = 0;
        const size_t want = c->arena_need + c->arena_need / 4;
        if (cudaMalloc((void**)&c->arena, want) == cudaSuccess) c->arena_cap = want;
        else (void)cudaGetLastError(); // no block: every array gets its own allocation, as on a first upload
    }
    c->arena_need = 0;

    Relayout R;
    if (const char* why = R.run(d)) return fail(c, VK_ERR_UNSUPPORTED, std::string("vk_scene_upload: ") + why);
    std::vector<vk_node>& nodes = R.nodes;
    std::vector<float4>& wnodes = R.wnodes;
    std::vector<vk_material> mats(d->materials, d->materials + d->n_materials);
    for (uint32_t i = 0; i < d->n_materials; ++i) {
        bool uv;
        if (mats[i].type == VK_M_SPECDIFFUSE)
            uv = (d->materials[mats[i].tex].type != VK_M_DIELECTRIC && v.tex_has_image(d->materials[mats[i].tex].tex, 0)) ||
                 (d->materials[mats[i].aux].type != VK_M_DIELECTRIC && v.tex_has_image(d->materials[mats[i].aux].tex, 0));
        else
            uv = mats[i].type != VK_M_DIELECTRIC && v.tex_has_image(mats[i].tex, 0);
        if (uv) mats[i].aux |= VKD_MAT_NEEDS_UV;
    }
    std::vector<float4> pvec((size_t)d->n_perlins * 256);
    std::vector<uint8_t> pperm((size_t)d->n_perlins * 768);
    for (uint32_t p = 0; p < d->n_perlins; ++p) {
        for (int k = 0; k < 256; ++k)
            pvec[(size_t)p * 256 + k] = make_float4(d->perlins[p].ranvec[k][0], d->perlins[p].ranvec[k][1], d->perlins[p].ranvec[k][2], 0.f);
        std::memcpy(&pperm[(size_t)p * 768], d->perlins[p].perm_x, 256);
        std::memcpy(&pperm[(size_t)p * 768 + 256], d->perlins[p].perm_y, 256);
        std::memcpy(&pperm[(size_t)p * 768 + 512], d->perlins[p].perm_z, 256);
    }

    // shading class per primitive, so that filing a finished traversal costs one byte load (vk_stepq.cu)
    std::vector<uint8_t> pcls;
    uint32_t cls_base[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    {
        auto cls_of = [&](uint32_t mat) -> uint8_t {
            const uint32_t t = mat < d->n_materials ? d->materials[mat].type : (uint32_t)VK_M_LAMBERTIAN;
            return t == VK_M_DIFFUSE_LIGHT ? 0 : t == VK_M_DIELECTRIC ? 1 : t == VK_M_METAL ? 2 : 3;
        };
        cls_base[VK_T_SPHERE] = (uint32_t)pcls.size();
        for (uint32_t i = 0; i < d->n_spheres; ++i) pcls.push_back(cls_of(d->sphere_mat[i]));
        cls_base[VK_T_MSPHERE] = (uint32_t)pcls.size();
        for (uint32_t i = 0; i < d->n_mspheres; ++i) pcls.push_back(cls_of(d->mspheres[i].mat));
        cls_base[VK_T_RECT] = (uint32_t)pcls.size();
        for (uint32_t i = 0; i < d->n_rects; ++i) pcls.push_back(cls_of(d->rects[i].mat));
        cls_base[VK_T_BOX] = (uint32_t)pcls.size();
        for (uint32_t i = 0; i < d->n_boxes; ++i) pcls.push_back(cls_of(d->boxes[i].mat));
        cls_base[VK_T_MEDIUM] = (uint32_t)pcls.size();
        for (uint32_t i = 0; i < d->n_media; ++i) pcls.push_back(cls_of(d->media[i].mat));
        pcls.push_back(3); // (never empty)
    }

    DScene s{};
    int rc;
#define UP(field, type, src, n)                                                                                        \
    if ((rc = upload<type>(c, (const type*)(src), (n), (const type**)&s.field)) != VK_OK) {                            \
        free_scene(c);                                                                                                 \
        return rc;                                                                                                     \
    }
    UP(wnodes, float4, wnodes.data(), wnodes.size())
    UP(nodes, float4, nodes.data(), (size_t)d->n_nodes * 2)
    UP(spheres, float4, d->spheres, d->n_spheres)
    UP(sphere_mat, uint32_t, d->sphere_mat, d->n_spheres)
    UP(mspheres, float4, d->mspheres, (size_t)d->n_mspheres * 3)
    UP(rects, float4, d->rects, (size_t)d->n_rects * 2)
    UP(boxes, float4, d->boxes, (size_t)d->n_boxes * 2)
    UP(xforms, float4, d->xforms, (size_t)d->n_xforms * 2)
    UP(media, float4, d->media, d->n_media)
    UP(media_plan, float4, R.media_plan.data(), R.media_plan.size())
    UP(lights, uint32_t, d->lights, d->n_lights)
    UP(materials, uint4, mats.data(), d->n_materials)
    UP(textures, uint4, d->textures, d->n_textures)
    UP(texels, uint8_t, d->texels, (size_t)d->n_texel_bytes)
    UP(perlin_vec, float4, pvec.data(), pvec.size())
    UP(perlin_perm, uint8_t, pperm.data(), pperm.size())
    UP(flat_shade, float4, R.flat_shade.data(), R.flat_shade.size())
    UP(prim_cls, uint8_t, pcls.data(), pcls.size())
#undef UP
    for (int t = 0; t < 8; ++t) s.cls_base[t] = cls_base[t];
    s.root = d->root;
    s.n_lights = d->n_lights;
    s.has_media = d->n_media > 0;
    s.light0_a = s.light0_b = make_float4(0.f, 0.f, 0.f, 0.f);
    if (d->n_lights >= 1 && VK_REF_TYPE(d->lights[0]) == VK_T_RECT) {
        static_assert(sizeof(vk_rect) == 2 * sizeof(float4), "device rect record");
        std::memcpy(&s.light0_a, &d->rects[VK_REF_INDEX(d->lights[0])], 2 * sizeof(float4));
    }
    CU(c, cudaStreamSynchronize(c->stream)); // host staging vectors die at return
    c->scene = s;
    c->n_nodes = d->n_nodes;
    c->n_materials = d->n_materials;
    c->n_textures = d->n_textures;
    c->n_media = d->n_media;
    c->wnodes_bytes = wnodes.size() * sizeof(float4);
    c->has_specdiffuse = R.has_specdiffuse;
    c->simple_scene = R.simple;
    c->flat_shape = R.flat_shape;
    c->one_rect_light = d->n_lights == 1 && VK_REF_TYPE(d->lights[0]) == VK_T_RECT && !(d->rects[VK_REF_INDEX(d->lights[0])].axes & VK_RECT_FLIP);
    c->stack_need = R.stack_need;
    c->levels_sub = R.levels_sub;
    c->flat = R.flat;
    c->has_scene = true;
    return VK_OK;
}

extern "C" int vk_flush_stats(vk_ctx* c, vk_stats* stats);

// Slot pool of the wavefront variant.  One allocation, carved into the arrays of WfState.  Default
// 2^19 slots: 96 B per slot = 50 MB, resident in the 126 MB L2, and
// 3-4 full waves of 256-thread CTAs per launch.  VECCHIO_WF_SLOTS overrides (tuning sweeps).
static int wf_ensure(vk_ctx* c) {
    uint32_t n = 1u << 19;
    if (const char* e = std::getenv("VECCHIO_WF_SLOTS")) {
        const long v = std::atol(e);
        if (v >= 1024 && v <= (1l << 26)) n = (uint32_t)v;
    }
    n = (n + 255u) & ~255u;
    if (c->wf_block && c->wf.n_slots == n) return VK_OK;
    if (c->wf_block) cudaFree(c->wf_block);
    c->wf_block = nullptr;
    c->wf = WfState{};
    const size_t per_slot = 16 * 5 + 4 * VKW_CLASSES;
    const size_t tail = 256; // qcount (2 sets) + unit_head
    CU(c, cudaMalloc(&c->wf_block, per_slot * n + tail));
    char* p = (char*)c->wf_block;
    auto take = [&](size_t bytes) { char* q = p; p += bytes; return q; };
    c->wf.ray_o = (float4*)take(16ull * n);
    c->wf.ray_d = (float4*)take(16ull * n);
    c->wf.beta = (float4*)take(16ull * n);
    c->wf.unit = (uint4*)take(16ull * n);
    c->wf.hit = (uint4*)take(16ull * n);
    c->wf.queue = (uint32_t*)take(4ull * VKW_CLASSES * n);
    c->wf.qcount = (uint32_t*)take(64);
    c->wf.unit_head = (unsigned long long*)take(64);
    c->wf.n_slots = n;
    if (!c->wf_host_counts) CU(c, cudaMallocHost((void**)&c->wf_host_counts, 64));
    return VK_OK;
}

// generate -> (extend -> shade)* until the pool has drained.  The host cannot see the pool, so it
// launches iterations in batches and reads the queue counters of the last extend after each batch
// (one 32-byte D2H + stream sync); an iteration on a drained pool is two empty launches.
static int wf_render(vk_ctx* c, bool strict, const FlatProgram* flat, const DCamera& dc, const RenderArgs& a, const RenderBuffers& b,
                     uint32_t* launches) {
    int rc = wf_ensure(c);
    if (rc != VK_OK) return rc;
    WfState w = c->wf;
    w.n_pixels = a.width * a.height;
    w.n_units = (unsigned long long)w.n_pixels * a.spp_count;
    const unsigned long long head0 = w.n_units < w.n_slots ? w.n_units : w.n_slots;
    CU(c, cudaMemsetAsync(w.qcount, 0, 64, c->stream));
    CU(c, cudaMemcpyAsync(w.unit_head, &head0, sizeof(head0), cudaMemcpyHostToDevice, c->stream));
    CU(c, strict ? vkstrict::launch_wf_generate(dc, a, w, c->stream) : vkfast::launch_wf_generate(dc, a, w, c->stream));
    ++*launches;
    // no sample ends before its first segment: at least spp_count * n_pixels / n_slots iterations
    const unsigned long long min_iters = ((unsigned long long)w.n_pixels * a.spp_count + w.n_slots - 1) / w.n_slots;
    unsigned long long next_check = min_iters > 8 ? min_iters : 8;
    const unsigned long long max_iters = (min_iters + 2) * (unsigned long long)a.max_depth + 64; // every path is <= max_depth segments
    for (unsigned long long it = 0;; ++it) {
        if (it > max_iters) {
            cudaStreamSynchronize(c->stream); // the kernels already launched still use the accumulators
            return fail(c, VK_ERR_CUDA, "wavefront: the slot pool did not drain (internal error)");
        }
        const uint32_t set = (uint32_t)(it & 1u);
        CU(c, strict ? vkstrict::launch_wf_extend(c->scene, flat, a, w, b, set, c->stream)
                     : vkfast::launch_wf_extend(c->scene, flat, a, w, b, set, c->stream));
        CU(c, strict ? vkstrict::launch_wf_shade(c->scene, dc, a, w, b, set, c->stream)
                     : vkfast::launch_wf_shade(c->scene, dc, a, w, b, set, c->stream));
        *launches += flat ? 2 : 3; // BVH scenes: extend + classify + shade
        if (it + 1 >= next_check) {
            CU(c, cudaMemcpyAsync(c->wf_host_counts, w.qcount + set * VKW_CLASSES, VKW_CLASSES * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
            CU(c, cudaStreamSynchronize(c->stream));
            const uint32_t live = c->wf_host_counts[0] + c->wf_host_counts[1] + c->wf_host_counts[2] + c->wf_host_counts[3];
            if (live == 0) break;
            // the pool is still busy: look again after about a quarter of what is left at most, at least 8 iterations
            next_check = it + 1 + (live == w.n_slots ? 32 : 8);
        }
    }
    return VK_OK;
}


// VK_VARIANT_AUTO, by the measurements recorded in profiles/ and DESIGN.md section 4:
//   scene small enough for the flat program  -> STAGED (Cornell 600x600x1000: 67 ms against 80 ms for
//       the lane megakernel and 138 ms for the global wavefront; 20 of 32 lanes active against 15,
//       instruction-fetch stalls gone)
//   BVH scenes                               -> MEGAKERNEL (final scene: 49 ms against 78 ms staged and
//       98 ms wavefront: while-while traversal diverges whatever the staging, and the lane
//       megakernel keeps 32 warps per SM against 24)
// (n_frames: a batch of frames is decided on its path count, all frames together)
static uint32_t choose_variant(const vk_ctx* c, const vk_render_params* P, uint32_t n_frames = 1) {
    if (P->variant != VK_VARIANT_AUTO) return P->variant;
    const bool flat = c->flat.n && !(P->flags & VK_FLAG_FORCE_BVH);
    // (a hybrid program holds subtrees whose traversal lengths vary: the lane megakernel, not the
    // barrier-synchronised staged kernel, runs it)
    const char* e = std::getenv("VECCHIO_AUTO"); // tuning sweeps: staged | warpq | mega
    if (e && !std::strcmp(e, "staged")) return flat && c->flat.n_bvh == 0 ? (uint32_t)VK_VARIANT_STAGED : (uint32_t)VK_VARIANT_MEGAKERNEL;
    if (e && !std::strcmp(e, "warpq")) return (uint32_t)VK_VARIANT_WARPQ;
    if (e && !std::strcmp(e, "stepq")) return flat && c->flat.n_bvh == 0 ? (uint32_t)VK_VARIANT_WARPQ : (uint32_t)VK_VARIANT_STEPQ;
    if (e && !std::strcmp(e, "mega")) return (uint32_t)VK_VARIANT_MEGAKERNEL;
    if (flat && c->flat.n_bvh == 0) return (uint32_t)VK_VARIANT_WARPQ;
    // BVH scenes: step queues where every leaf sits in the world frame (random spheres 8.9 against 10.7 ms, 10^6 spheres 23.7
    // against 29.0 ms); scenes with instanced sub-BVHs (final scene: 50.6 against 45.8 ms) stay on the lane megakernel
    // -- and only for frames that fill the pools a few dozen times over: 227 000 slots are resident, and below ~3 M paths
    // their start-up and drain cost more than the fuller warps gain (random spheres 400x225: 16 spp 1.32 against 1.21 ms,
    // 32 spp 1.85 against 1.83, 64 spp 2.78 against 3.30; profiles/r2_sweep_9.log)
    const uint64_t paths = (uint64_t)P->width * P->height * (P->spp_count ? P->spp_count : P->spp - P->spp_begin) * n_frames;
    return c->levels_sub == 0u && paths >= (4ull << 20) ? (uint32_t)VK_VARIANT_STEPQ : (uint32_t)VK_VARIANT_MEGAKERNEL;
}

// Lane megakernel for a BVH scene: static (one whole ray per lane and loop iteration) or dynamic
// (resumable traversal under warp votes with re-fill).  Measured on B200 (profiles/r1_configs_dyn.log):
// the dynamic kernel wins where traversal lengths have a long tail -- 10^6 spheres, 66 node visits per
// ray: 62 ms against 96 ms, 15.6 against 4.5 lanes active -- and loses on the small heterogeneous
// scenes (final scene 57 ms against 44 ms, random spheres 13.8 against 13.1 ms), where shading is a
// larger share of the work and runs with few lanes during a re-fill.  VECCHIO_MEGA=static|dynamic overrides.
static bool use_dynamic_megakernel(const vk_ctx* c) {
    if (const char* e = std::getenv("VECCHIO_MEGA")) {
        if (!std::strcmp(e, "static")) return false;
        if (!std::strcmp(e, "dynamic")) return true;
    }
    return c->n_nodes >= 65536u;
}

// Large BVHs (the 10^6-sphere scene: 64 MB of 4-wide nodes, every ray touches ~30 of them at random) share the
// 126 MB L2 with the frame's accumulators (a 4K frame is 199 MB of atomics streaming through).  An access-policy window
// on the node array keeps the nodes' lines resident (persisting) and lets everything else stream.  Small scenes are
// L1 / L2 resident anyway and get no window.  VECCHIO_L2_PERSIST=0 turns it off (A/B runs).
static void apply_l2_window(vk_ctx* c) {
    cudaStreamAttrValue v{};
    const char* e = std::getenv("VECCHIO_L2_PERSIST");
    const bool on = c->wnodes_bytes >= (8u << 20) && c->l2_persist_max && c->l2_window_max && !(e && e[0] == '0');
    if (on) {
        const size_t bytes = c->wnodes_bytes < c->l2_window_max ? c->wnodes_bytes : c->l2_window_max;
        v.accessPolicyWindow.base_ptr = (void*)c->scene.wnodes;
        v.accessPolicyWindow.num_bytes = bytes;
        v.accessPolicyWindow.hitRatio = bytes <= c->l2_persist_max ? 1.0f : (float)((double)c->l2_persist_max / (double)bytes);
        v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    } // else: a zero-sized window clears a previous scene's
    cudaStreamSetAttribute(c->stream, cudaStreamAttributeAccessPolicyWindow, &v);
    cudaGetLastError();
}

// The staged and wavefront kernels render one whole frame per launch: no batches of frames, no pixel lists (list: an
// adaptive render's passes).  `variant`: the one asked for, or the one AUTO chose.
static int check_variant(vk_ctx* c, const std::string& who, uint32_t variant, uint32_t n_frames, bool list) {
    if (variant != VK_VARIANT_STAGED && variant != VK_VARIANT_WAVEFRONT) return VK_OK;
    if (list) return fail(c, VK_ERR_UNSUPPORTED, who + ": the staged and wavefront kernels have no pixel-list passes");
    if (n_frames > 1) return fail(c, VK_ERR_UNSUPPORTED, who + ": the staged and wavefront kernels render one frame per call");
    return VK_OK;
}

// What every render call refuses of its cameras and parameters before anything is allocated or launched (`who` names the
// call in the message).  adaptive: a render in passes over pixel lists (vk_render_adaptive*, vk_adaptive_begin*), with its
// pass_spp and the one-shot calls' max_error (a session checks its targets in refine).
static int check_render(vk_ctx* c, const std::string& who, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P,
                        bool adaptive = false, uint32_t pass_spp = 0, float max_error = 0.0f) {
    if (!cams || !P || n_frames == 0) return fail(c, VK_ERR_INVALID, who + ": null argument or no frames");
    if (!c->has_scene) return fail(c, VK_ERR_NO_SCENE, who + ": no scene uploaded");
    if (P->width < 2 || P->height < 2) return fail(c, VK_ERR_INVALID, who + ": width/height must be >= 2 ((width-1) divides, src/main.rs:187)");
    if (P->spp == 0 || P->spp_begin >= P->spp) return fail(c, VK_ERR_INVALID, who + ": bad spp / spp_begin");
    // the kernels trace a path's first segment before they test its depth; depth 0 is a black frame with no rays
    if (P->max_depth == 0) return fail(c, VK_ERR_INVALID, who + ": max_depth must be >= 1 (ray_color starts at depth 1, src/main.rs:126)");
    const uint32_t count = P->spp_count ? P->spp_count : P->spp - P->spp_begin;
    if ((uint64_t)P->spp_begin + count > P->spp) return fail(c, VK_ERR_INVALID, who + ": sample slice exceeds spp");
    // the kernels index the accumulators of the whole batch with 32-bit element indices
    if ((uint64_t)P->width * P->height * n_frames > 0x7FFFFFFFull / 3)
        return fail(c, VK_ERR_INVALID, who + ": image too large (n_frames * width * height * 3 exceeds 2^31 - 1)");
    if (P->variant > VK_VARIANT_STEPQ) return fail(c, VK_ERR_INVALID, who + ": unknown variant");
    for (uint32_t f = 0; f < n_frames; ++f)
        if (!(cams[f].time0 < cams[f].time1))
            return fail(c, VK_ERR_INVALID, who + ": frame " + std::to_string(f) + ": camera time0 >= time1 (gen_range panics, src/main.rs:118)");
    if (adaptive) {
        if (pass_spp == 0) return fail(c, VK_ERR_INVALID, who + ": pass_spp must be >= 1");
        if (!(max_error >= 0.0f)) return fail(c, VK_ERR_INVALID, who + ": max_error must be >= 0 (and not NaN)");
        if (P->spp_begin != 0 || (P->spp_count != 0 && P->spp_count != P->spp))
            return fail(c, VK_ERR_INVALID, who + ": an adaptive render draws samples [0, n_p) of every pixel: spp_begin must be 0, spp_count 0 or spp");
        if (P->spp > VK_ADAPTIVE_MAX_SPP)
            return fail(c, VK_ERR_INVALID, who + ": spp above " + std::to_string(VK_ADAPTIVE_MAX_SPP) +
                                               ", the limit of the fixed-point sums of squares (2^16 samples of at most 255^2 * 2^32 units)");
    }
    return check_variant(c, who, P->variant, n_frames, adaptive);
}

// The kernel a call runs and how it is launched, decided once per call (an adaptive render runs every pass on it).
struct RenderPlan {
    bool strict, legacy, l0;
    const FlatProgram* flat;
    uint32_t variant;
    int grid;
    uint32_t resident_warps;
};
// (check_render has passed; list: the passes of an adaptive render)
static int plan_render(vk_ctx* c, const std::string& who, const vk_render_params* P, uint32_t n_frames, bool list, RenderPlan* R) {
    R->strict = (P->flags & VK_FLAG_STRICT_MATH) != 0;
    const bool strict = R->strict;
    const FlatProgram* flat = (c->flat.n && !(P->flags & VK_FLAG_FORCE_BVH)) ? &c->flat : nullptr;
    int bps = 0, bt = 0;
    const bool legacy = (P->flags & VK_FLAG_LEGACY_SCATTER) != 0;
    uint32_t variant = choose_variant(c, P, n_frames);
    if (legacy && variant != VK_VARIANT_WARPQ && variant != VK_VARIANT_STEPQ) variant = VK_VARIANT_MEGAKERNEL; // legacy integrator: lane megakernel and warp queues
    // a hybrid program (flat top + homogeneous subtrees) is the warp-queue kernel's: every other variant walks the BVH
    // (lane megakernel on it: 51.5 against 46.1 ms on the final scene, profiles/r2_sweep_12.log)
    if (flat && flat->n_bvh && variant != VK_VARIANT_WARPQ && !std::getenv("VECCHIO_HYBRID_ALL")) flat = nullptr;
    if (legacy && c->has_specdiffuse)
        return fail(c, VK_ERR_UNSUPPORTED, who + ": SpecDiffuse has no legacy scatter (the reference's default unwraps a missing specular ray and panics, src/material.rs:21-28)");
    if (!legacy && c->scene.n_lights == 0)
        return fail(c, VK_ERR_INVALID, who + ": empty light list (the reference panics: choose().unwrap(), src/hittable.rs:431); only VK_FLAG_LEGACY_SCATTER renders without lights");
    if (const int rc = check_variant(c, who, variant, n_frames, list); rc != VK_OK) return rc;
    // the render build compiled for a light list of one unflipped Rect (VK_LIGHT0, see vk_device.cuh)
    const bool l0 = !strict && !legacy && c->one_rect_light && !c->has_specdiffuse && !std::getenv("VECCHIO_NO_LIGHT0");
    CU(c, strict ? vkstrict::megakernel_occupancy(flat != nullptr, c->scene.has_media, legacy, &bps, &bt)
          : l0   ? vkfast_l0::megakernel_occupancy(flat != nullptr, c->scene.has_media, legacy, &bps, &bt)
                 : vkfast::megakernel_occupancy(flat != nullptr, c->scene.has_media, legacy, &bps, &bt));
    if (bps < 1) bps = 1;
    R->legacy = legacy;
    R->l0 = l0;
    R->flat = flat;
    R->grid = c->sm_count * bps;
    R->resident_warps = (uint32_t)R->grid * (uint32_t)bt / 32u;
    if (variant == VK_VARIANT_STEPQ && flat && flat->n_bvh == 0) variant = VK_VARIANT_WARPQ; // step queues are the BVH traversal; a flat program has none
    R->variant = variant;
    return VK_OK;
}

// A batch's cameras go to the device with each launch over it (the kernels read them at regeneration only): c->cams.
static int upload_cams(vk_ctx* c, const vk_camera* cams, uint32_t n_frames) {
    if (c->cams_cap < n_frames) {
        if (c->cams) cudaFree(c->cams);
        c->cams = nullptr;
        c->cams_cap = 0;
        CU(c, cudaMalloc((void**)&c->cams, n_frames * sizeof(DCamera)));
        c->cams_cap = n_frames;
    }
    c->cams_host.resize(n_frames);
    for (uint32_t f = 0; f < n_frames; ++f) c->cams_host[f] = to_dcam(cams + f);
    CU(c, cudaMemcpyAsync(c->cams, c->cams_host.data(), n_frames * sizeof(DCamera), cudaMemcpyHostToDevice, c->stream));
    return VK_OK;
}

// One launch of the sample loop over global samples [spp_begin, spp_begin + count) into the accumulators of b (which the
// caller has zeroed), on the kernel R names.  The work domain: n_frames > 1, cam points to n_frames cameras (FrameArgs);
// ls != nullptr, only the listed pixels of one frame (ListArgs), or with n_frames > 1 of the batch (FrameListArgs: the
// entries are batch-wide pixels); otherwise one frame (OneFrame).  Adds the kernels it launched to *launches.
static int launch_pass(vk_ctx* c, const RenderPlan& R, const vk_camera* cam, const vk_render_params* P, uint32_t spp_begin, uint32_t count,
                       const RenderBuffers& b, uint32_t n_frames, const ListArgs* ls, uint32_t* launches) {
    const bool strict = R.strict, legacy = R.legacy, l0 = R.l0;
    const FlatProgram* flat = R.flat;
    const uint32_t variant = R.variant;
    RenderArgs a{};
    a.width = P->width;
    a.height = P->height;
    a.spp_begin = spp_begin;
    a.spp_count = count;
    a.max_depth = P->max_depth;
    a.seed_lo = (uint32_t)P->seed;
    a.seed_hi = (uint32_t)(P->seed >> 32);
    a.background = make_float3(P->background[0], P->background[1], P->background[2]);
    a.flags = P->flags;
    a.tiles_x = (P->width + 7) / 8;
    a.tiles_y = (P->height + 3) / 4;
    if (ls) { // the lane megakernel's items over a list: groups of 32 consecutive entries
        a.tiles_x = (ls->n + 31) / 32;
        a.tiles_y = 1;
    }
    // Lane megakernel: chunks of samples, sized for ~48 work items per resident warp (small items keep
    // the end-of-kernel tail short; an item costs one atomic).
    // (a batch: the items of all its frames share the warps; a list across frames already spans them)
    const uint32_t n_tiles = a.tiles_x * a.tiles_y * (ls ? 1u : n_frames);
    uint32_t n_chunks = (48u * R.resident_warps + n_tiles - 1) / n_tiles;
    if (n_chunks > count) n_chunks = count;
    if (n_chunks < 1) n_chunks = 1;
    a.chunk_spp = (count + n_chunks - 1) / n_chunks;
    a.n_chunks = (count + a.chunk_spp - 1) / a.chunk_spp;

    CU(c, cudaMemsetAsync(c->counters + 2, 0, sizeof(unsigned long long), c->stream)); // work-queue head only
    const DCamera dc = to_dcam(cam);
    // the variant switch, for the work domain `dom` (staged and wavefront have none: check_variant keeps batches and pixel
    // lists away from them)
    auto run = [&](const auto& dom) -> int {
        if (variant == VK_VARIANT_STEPQ) {
            const bool inst = c->levels_sub != 0u;
            uint32_t glevels = 0;
            const size_t words = strict ? vkstrict::stepq_stack_words(c->stack_need, inst, c->sm_count, &glevels)
                                        : vkfast::stepq_stack_words(c->stack_need, inst, c->sm_count, &glevels);
            if (words) {
                const int rc = ensure(c, &c->sq_stack, &c->sq_stack_floats, words);
                if (rc != VK_OK) return rc;
            }
            CU(c, cudaMemsetAsync(c->counters + 2, 0, sizeof(unsigned long long), c->stream)); // unit queue head
            CU(c, cudaMemsetAsync(c->counters + 5, 0, sizeof(unsigned long long), c->stream)); // self-check violations (debug builds)
            CU(c, strict ? vkstrict::launch_stepq(c->scene, dc, a, b, c->counters + 2, (uint32_t*)c->sq_stack, glevels, inst, c->sm_count, legacy, c->stream, dom)
                  : l0   ? vkfast_l0::launch_stepq(c->scene, dc, a, b, c->counters + 2, (uint32_t*)c->sq_stack, glevels, inst, c->sm_count, legacy, c->stream, dom)
                         : vkfast::launch_stepq(c->scene, dc, a, b, c->counters + 2, (uint32_t*)c->sq_stack, glevels, inst, c->sm_count, legacy, c->stream, dom));
            *launches += 1;
        } else if (variant == VK_VARIANT_WARPQ) {
            CU(c, cudaMemsetAsync(c->counters + 2, 0, sizeof(unsigned long long), c->stream)); // unit queue head
            CU(c, cudaMemsetAsync(c->counters + 5, 0, sizeof(unsigned long long), c->stream)); // self-check violations (debug builds)
            // (a hybrid program -- flat top, homogeneous subtrees walked inside extend -- runs k_warpq_hybrid)
            const FlatProgram* sflat = flat;
            const bool simple = !strict && !legacy && sflat && sflat->n_bvh == 0 && c->simple_scene && !std::getenv("VECCHIO_NO_SIMPLE");
            // the trimmed build's kernel compiled for the program's shape, if there is one (VECCHIO_NO_STATIC_FLAT: the generic one)
            const uint32_t shape = std::getenv("VECCHIO_NO_STATIC_FLAT") ? (uint32_t)VKF_SHAPE_NONE : c->flat_shape;
            CU(c, strict   ? vkstrict::launch_warpq(c->scene, sflat, VKF_SHAPE_NONE, dc, a, b, c->counters + 2, c->sm_count, legacy, c->stream, dom)
                  : simple ? vkfast_simple::launch_warpq(c->scene, sflat, shape, dc, a, b, c->counters + 2, c->sm_count, legacy, c->stream, dom)
                  : l0     ? vkfast_l0::launch_warpq(c->scene, sflat, VKF_SHAPE_NONE, dc, a, b, c->counters + 2, c->sm_count, legacy, c->stream, dom)
                           : vkfast::launch_warpq(c->scene, sflat, VKF_SHAPE_NONE, dc, a, b, c->counters + 2, c->sm_count, legacy, c->stream, dom));
            *launches += 1;
        } else if (variant == VK_VARIANT_WAVEFRONT) {
            uint32_t n = 0;
            int rc = wf_render(c, strict, flat, dc, a, b, &n);
            if (rc != VK_OK) return rc;
            *launches += n;
        } else if (variant == VK_VARIANT_STAGED) {
            CU(c, cudaMemsetAsync(c->counters + 5, 0xFF, 2 * sizeof(unsigned long long), c->stream)); // CTA start / first end: minima
            CU(c, cudaMemsetAsync(c->counters + 7, 0, sizeof(unsigned long long), c->stream));        // last end: maximum
            CU(c, cudaMemsetAsync(c->counters + 2, 0, sizeof(unsigned long long), c->stream)); // unit queue head
            // a "simple" scene runs the build of the same kernel with the unreachable code compiled out
            // (the staged kernel's K-ray flat trace has no subtree entries: a hybrid program means its BVH path)
            const FlatProgram* sflat = flat && flat->n_bvh == 0 ? flat : nullptr;
            const bool simple = !strict && sflat && c->simple_scene && !std::getenv("VECCHIO_NO_SIMPLE");
            CU(c, strict   ? vkstrict::launch_staged(c->scene, sflat, dc, a, b, c->counters + 2, c->sm_count, c->stream)
                  : simple ? vkfast_simple::launch_staged(c->scene, sflat, dc, a, b, c->counters + 2, c->sm_count, c->stream)
                           : vkfast::launch_staged(c->scene, sflat, dc, a, b, c->counters + 2, c->sm_count, c->stream));
            *launches += 1;
        } else if (!flat && !legacy && use_dynamic_megakernel(c)) {
            CU(c, cudaMemsetAsync(c->counters + 2, 0, sizeof(unsigned long long), c->stream)); // unit queue head
            CU(c, strict ? vkstrict::launch_megakernel_dyn(c->scene, dc, a, b, c->counters + 2, c->sm_count, c->stream, dom)
                  : l0   ? vkfast_l0::launch_megakernel_dyn(c->scene, dc, a, b, c->counters + 2, c->sm_count, c->stream, dom)
                         : vkfast::launch_megakernel_dyn(c->scene, dc, a, b, c->counters + 2, c->sm_count, c->stream, dom));
            *launches += 1;
        } else {
            CU(c, strict ? vkstrict::launch_megakernel(c->scene, flat, dc, a, b, R.grid, legacy, c->stream, dom)
                  : l0   ? vkfast_l0::launch_megakernel(c->scene, flat, dc, a, b, R.grid, legacy, c->stream, dom)
                         : vkfast::launch_megakernel(c->scene, flat, dc, a, b, R.grid, legacy, c->stream, dom));
            *launches += 1;
        }
        return VK_OK;
    };
    if (n_frames == 1) return ls ? run(*ls) : run(OneFrame{});
    int rc = upload_cams(c, cam, n_frames);
    if (rc != VK_OK) return rc;
    const FrameArgs fr{c->cams, n_frames, P->width * P->height};
    return ls ? run(FrameListArgs{fr, *ls}) : run(fr);
}

// shared body of vk_render / vk_render_device / vk_render_frames*
// acc_only: leave the result in the context's integer accumulators (c->partial) and skip the conversion to fp32 sums
// (the multi-GPU context reduces the accumulators of all its devices itself); want_sq then says whether squares are kept
// n_frames > 1: cam points to n_frames cameras and the result is n_frames contiguous planes (the batch kernels take
// FrameArgs, everything else is the single-frame path)
static int render_into(vk_ctx* c, const vk_camera* cam, const vk_render_params* P, float* d_sum, float* d_sumsq, vk_stats* stats,
                       bool acc_only = false, bool want_sq = false, uint32_t n_frames = 1) {
    if (!c) return VK_ERR_INVALID;
    int rc = check_render(c, "render", cam, n_frames, P);
    if (rc != VK_OK) return rc;
    if (!d_sum && !acc_only) return fail(c, VK_ERR_INVALID, "render: null argument");
    if (!acc_only) want_sq = d_sumsq != nullptr;
    const uint32_t count = P->spp_count ? P->spp_count : P->spp - P->spp_begin;
    CU(c, cudaSetDevice(c->device));
    RenderPlan R;
    if ((rc = plan_render(c, "render", P, n_frames, false, &R)) != VK_OK) return rc;

    // Accumulators (see RenderBuffers): u64 fixed-point sums, plus double sums of squares when asked for.
    const size_t plane = (size_t)P->width * P->height * 3 * n_frames;
    RenderBuffers b{};
    b.counters = c->counters;
    b.debug = c->debug;
    {
        rc = ensure(c, &c->partial, &c->partial_floats, plane * (want_sq ? 4 : 2));
        if (rc != VK_OK) return rc;
        b.acc = (unsigned long long*)c->partial;
        b.accsq = want_sq ? (double*)(c->partial + plane * 2) : nullptr;
        CU(c, cudaMemsetAsync(c->partial, 0, plane * (want_sq ? 4 : 2) * sizeof(float), c->stream));
    }
    apply_l2_window(c);
    CU(c, cudaEventRecord(c->ev0, c->stream));
    uint32_t launches = 0;
    if ((rc = launch_pass(c, R, cam, P, P->spp_begin, count, b, n_frames, nullptr, &launches)) != VK_OK) return rc;
    if (!acc_only) {
        k_acc_to_sum<<<(unsigned)((plane + 255) / 256), 256, 0, c->stream>>>(b.acc, b.accsq, plane, d_sum, d_sumsq);
        ++launches;
    }
    CU(c, cudaGetLastError());
    CU(c, cudaEventRecord(c->ev1, c->stream));
    c->launches += launches;
    c->paths += (uint64_t)P->width * P->height * count * n_frames;
    if (stats) { // reading the counters synchronises; with stats == NULL the call is fully asynchronous
        rc = vk_flush_stats(c, stats);
        if (rc != VK_OK) return rc;
        CU(c, cudaEventElapsedTime(&stats->ms_kernels, c->ev0, c->ev1));
        stats->ms_total = stats->ms_kernels;
        stats->variant = R.variant;
    }
    return VK_OK;
}

int vk_render_device(vk_ctx* c, const vk_camera* cam, const vk_render_params* P, float* d_sum, float* d_sumsq, vk_stats* stats) {
    return render_into(c, cam, P, d_sum, d_sumsq, stats);
}

int vk_finalize_device(vk_ctx* c, const float* d_sum, float* d_rgb, size_t n, uint32_t spp) {
    if (!c || !d_sum || !d_rgb || spp == 0) return fail(c, VK_ERR_INVALID, "vk_finalize_device: bad argument");
    CU(c, cudaSetDevice(c->device));
    if (n) k_finalize<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(SumsOverSpp{d_sum, (float)spp}, d_rgb, n);
    c->launches += n ? 1 : 0;
    CU(c, cudaGetLastError());
    return VK_OK;
}

int vk_set_stream(vk_ctx* c, void* stream) {
    if (!c) return VK_ERR_INVALID;
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaStreamSynchronize(c->stream));
    c->stream = stream ? (cudaStream_t)stream : c->own_stream;
    return VK_OK;
}

int vk_flush_stats(vk_ctx* c, vk_stats* stats) {
    if (!c || !stats) return VK_ERR_INVALID;
    CU(c, cudaSetDevice(c->device));
    unsigned long long h[5] = {0, 0, 0, 0, 0};
    CU(c, cudaMemcpyAsync(h, c->counters, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemsetAsync(c->counters, 0, 2 * sizeof(unsigned long long), c->stream));
    CU(c, cudaMemsetAsync(c->counters + 3, 0, 2 * sizeof(unsigned long long), c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    std::memset(stats, 0, sizeof(*stats));
    stats->paths = c->paths;
    stats->rays = h[0];
    stats->dropped_samples = h[1];
    stats->node_visits = h[3];
    stats->prim_tests = h[4];
    stats->launches = (uint32_t)c->launches;
    stats->variant = VK_VARIANT_MEGAKERNEL;
    c->paths = 0;
    c->launches = 0;
    return VK_OK;
}

// Device state of a session: fixed-point sums and squares and the counts of every pixel of its K frames, plus the pass
// loop's scratch (two pixel lists, the select flags, the level of every pixel, the level counts, the compaction scratch).
struct vk_adaptive_session {
    vk_ctx* c = nullptr;
    std::vector<vk_camera> cams;
    vk_render_params P{}; // P.spp: the session's limit
    uint32_t n_frames = 0, pass_spp = 0, n_pix = 0, max_levels = 0;
    uint32_t shard = 0, n_shards = 1, n_owned = 0; // the pixels the pass loop renders: shard_owns(p, shard, n_shards), n_owned of them
    RenderPlan R{};
    uint64_t scene_gen = 0;
    bool reached_any = false; // a target has been reached (or imported); false: every count is 0
    bool broken = false;      // a refine or import failed on the device part way: the state is lost
    vk_adaptive_target reached{};
    void* block = nullptr;
    size_t bytes = 0, cub_bytes = 0;
    unsigned long long *acc = nullptr, *sq = nullptr;
    uint32_t *nspp = nullptr, *cur = nullptr, *nxt = nullptr, *level = nullptr, *n_level = nullptr;
    uint8_t* keep = nullptr;
    int* d_count = nullptr;
    void* cub_tmp = nullptr;
};

// What a render call hands back to host buffers (null: not asked for): the image as floats or as rgb8 bytes, a fixed
// render's sums of squares, an adaptive read's counts and error map.
struct Outputs {
    float* rgb;
    uint8_t* rgb8;
    float* sumsq;
    uint32_t* spp;
    float* error;
};

// Where a call's results lie in c->frame and c->pinned, in floats from the start of each: the image, the squares, the counts
// and the error map at the same offsets on both sides, then on the device only the float sums of a fixed render (`fixed`).
// A fixed render stages before its sums are written, so that the readout's own call finds the buffers large enough and
// moves nothing.
struct Staging {
    size_t sumsq, counts, error, sum;
};
static int stage(vk_ctx* c, size_t plane, bool fixed, const Outputs& o, Staging* S) {
    const size_t n_pix = plane / 3;
    S->sumsq = o.rgb ? plane : (plane + 3) / 4;
    S->counts = S->sumsq + (o.sumsq ? plane : 0);
    S->error = S->counts + (o.spp ? n_pix : 0);
    S->sum = S->error + (o.error ? n_pix : 0);
    const int rc = ensure(c, &c->frame, &c->frame_floats, S->sum + (fixed ? plane : 0));
    return rc != VK_OK ? rc : ensure_pinned(c, S->sum);
}

// The chunked copy-out every call into host buffers ends with: n elements of elem bytes from the start of c->frame go to the
// host through c->pinned in VK_CHUNKS chunks.  chunks_begin enqueues the copies (off: the chunks' byte offsets); chunks_end
// waits for each chunk in turn and hands its bytes to the caller's buffers it covers, so that they fill from one chunk while
// the later ones are still on the bus.
#define VK_CHUNKS 4
struct HostSpan { // bytes [begin, end) of the staged result are host[0 .. end - begin)
    char* host;
    size_t begin, end;
};
static int chunks_begin(vk_ctx* c, size_t n, size_t elem, size_t off[VK_CHUNKS + 1]) {
    for (int i = 0; i <= VK_CHUNKS; ++i) off[i] = n * (size_t)i / VK_CHUNKS * elem;
    for (int i = 0; i < VK_CHUNKS; ++i) {
        if (!c->ev_chunk[i]) CU(c, cudaEventCreateWithFlags(&c->ev_chunk[i], cudaEventDisableTiming));
        CU(c, cudaMemcpyAsync((char*)c->pinned + off[i], (const char*)c->frame + off[i], off[i + 1] - off[i], cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaEventRecord(c->ev_chunk[i], c->stream));
    }
    return VK_OK;
}
static int chunks_end(vk_ctx* c, const size_t off[VK_CHUNKS + 1], const HostSpan* spans, int n_spans) {
    for (int i = 0; i < VK_CHUNKS; ++i) {
        CU(c, cudaEventSynchronize(c->ev_chunk[i]));
        for (int k = 0; k < n_spans; ++k) {
            const size_t b = off[i] > spans[k].begin ? off[i] : spans[k].begin, e = off[i + 1] < spans[k].end ? off[i + 1] : spans[k].end;
            if (b < e) std::memcpy(spans[k].host + (b - spans[k].begin), (const char*)c->pinned + b, e - b);
        }
    }
    return VK_OK;
}

// The end of every render call into host buffers, given its result on c's device: the float sums over P->spp of a fixed
// render (s == nullptr) in c->frame where stage() puts them, or session s's state.  Converts the means of the n_frames
// frames into c->frame (k_finalize, or k_to_color with the counts in the image's order), copies the image back through
// c->pinned in four chunks -- the caller's buffer fills from each chunk while the later ones are still on the bus -- and the
// extras whole, records ev1 and synchronises.  With stats, adds the readout's launches and ends ms_total at ev1 (it began
// at ev2).
static int readout(vk_ctx* c, const vk_render_params* P, uint32_t n_frames, const vk_adaptive_session* s, const Outputs& o, vk_stats* stats) {
    const size_t plane = (size_t)P->width * P->height * 3 * n_frames, n_pix = plane / 3;
    CU(c, cudaSetDevice(c->device));
    Staging S;
    int rc = stage(c, plane, !s, o, &S);
    if (rc != VK_OK) return rc;
    float* d = c->frame;
    uint32_t* d_spp = o.spp && o.rgb8 ? (uint32_t*)(d + S.counts) : nullptr; // (a float image's counts: the session's own, in pixel order)
    auto convert = [&](auto src) {
        const unsigned blocks = (unsigned)((plane + 255) / 256);
        if (o.rgb) k_finalize<<<blocks, 256, 0, c->stream>>>(src, d, plane);
        else k_to_color<<<blocks, 256, 0, c->stream>>>(src, (uint8_t*)d, d_spp, P->width, P->height, n_frames);
    };
    if (s) convert(AccOverCount{s->acc, s->nspp});
    else convert(SumsOverSpp{d + S.sum, (float)P->spp});
    CU(c, cudaGetLastError());
    size_t off[VK_CHUNKS + 1];
    if ((rc = chunks_begin(c, plane, o.rgb ? sizeof(float) : 1, off)) != VK_OK) return rc;
    if (o.sumsq) CU(c, cudaMemcpyAsync(c->pinned + S.sumsq, d + S.sumsq, plane * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    if (o.spp) CU(c, cudaMemcpyAsync(c->pinned + S.counts, d_spp ? d_spp : s->nspp, n_pix * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    if (o.error) {
        k_adaptive_error_map<<<(unsigned)((n_pix + 255) / 256), 256, 0, c->stream>>>(s->acc, s->sq, s->nspp, d + S.error, P->width, P->height,
                                                                                     n_frames, o.rgb8 != nullptr);
        CU(c, cudaGetLastError());
        CU(c, cudaMemcpyAsync(c->pinned + S.error, d + S.error, n_pix * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    }
    CU(c, cudaEventRecord(c->ev1, c->stream));
    const HostSpan image{o.rgb ? (char*)o.rgb : (char*)o.rgb8, 0, off[VK_CHUNKS]};
    if ((rc = chunks_end(c, off, &image, 1)) != VK_OK) return rc;
    CU(c, cudaStreamSynchronize(c->stream));
    if (o.sumsq) std::memcpy(o.sumsq, c->pinned + S.sumsq, plane * sizeof(float));
    if (o.spp) std::memcpy(o.spp, c->pinned + S.counts, n_pix * sizeof(uint32_t));
    if (o.error) std::memcpy(o.error, c->pinned + S.error, n_pix * sizeof(float));
    if (stats) {
        stats->launches += o.error ? 2 : 1;
        c->launches = 0;
        CU(c, cudaEventElapsedTime(&stats->ms_total, c->ev2, c->ev1));
    }
    return VK_OK;
}

// shared body of vk_render, vk_render_rgb8, vk_render_frames and vk_render_frames_rgb8: one launch over every frame's units
// into float sums (and squares) in c->frame, then the readout
static int render_host(vk_ctx* c, const std::string& who, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P, float* out_rgb,
                       uint8_t* out_rgb8, float* out_sumsq, vk_stats* stats) {
    if (!c) return VK_ERR_INVALID;
    if (!out_rgb && !out_rgb8) return fail(c, VK_ERR_INVALID, who + ": null argument");
    int rc = check_render(c, who, cams, n_frames, P);
    if (rc != VK_OK) return rc;
    const Outputs o{out_rgb, out_rgb8, out_sumsq, nullptr, nullptr};
    CU(c, cudaSetDevice(c->device));
    Staging S;
    if ((rc = stage(c, (size_t)P->width * P->height * 3 * n_frames, true, o, &S)) != VK_OK) return rc;
    CU(c, cudaEventRecord(c->ev2, c->stream));
    vk_stats st{};
    rc = render_into(c, cams, P, c->frame + S.sum, out_sumsq ? c->frame + S.sumsq : nullptr, &st, false, false, n_frames);
    if (rc == VK_OK) rc = readout(c, P, n_frames, nullptr, o, &st);
    if (rc == VK_OK && stats) *stats = st;
    return rc;
}

int vk_render(vk_ctx* c, const vk_camera* cam, const vk_render_params* P, float* out_rgb, float* out_sumsq, vk_stats* stats) {
    return render_host(c, "vk_render", cam, 1, P, out_rgb, nullptr, out_sumsq, stats);
}

int vk_render_rgb8(vk_ctx* c, const vk_camera* cam, const vk_render_params* P, uint8_t* out_rgb8, vk_stats* stats) {
    return render_host(c, "vk_render_rgb8", cam, 1, P, nullptr, out_rgb8, nullptr, stats);
}

int vk_render_frames(vk_ctx* c, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P, float* out_rgb, vk_stats* stats) {
    return render_host(c, "vk_render_frames", cams, n_frames, P, out_rgb, nullptr, nullptr, stats);
}

int vk_render_frames_rgb8(vk_ctx* c, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P, uint8_t* out_rgb8, vk_stats* stats) {
    return render_host(c, "vk_render_frames_rgb8", cams, n_frames, P, nullptr, out_rgb8, nullptr, stats);
}

// The traversal vk_intersect and vk_render_aov run: the flat program, unless it holds subtrees (a hybrid program is the
// warp-queue kernel's) or the flags force the BVH; nullptr: the BVH
static const FlatProgram* hit_program(const vk_ctx* c, uint32_t flags) {
    return (c->flat.n && (c->flat.n_bvh == 0 || std::getenv("VECCHIO_HYBRID_ALL")) && !(flags & VK_FLAG_FORCE_BVH)) ? &c->flat : nullptr;
}

// shared body of vk_render_aov and vk_multi_render_aov: one k_aov launch writes the planes asked for, packed in the order
// albedo, normal, depth, coverage, into c->frame (staged as one float image), then the chunked copy-out hands each to its buffer
static int render_aov(vk_ctx* c, const std::string& who, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P, uint32_t aov_spp,
                      float* out_albedo, float* out_normal, float* out_depth, float* out_coverage, vk_stats* stats) {
    if (!c) return VK_ERR_INVALID;
    vk_render_params q{}; // every check of vk_render_frames but the variant's: no render kernel runs
    if (P) {
        q = *P;
        q.variant = VK_VARIANT_AUTO;
    }
    int rc = check_render(c, who, cams, n_frames, P ? &q : nullptr);
    if (rc != VK_OK) return rc;
    if (aov_spp == 0 || aov_spp > VK_AOV_MAX_SPP) return fail(c, VK_ERR_INVALID, who + ": aov_spp must be 1 .. " + std::to_string(VK_AOV_MAX_SPP));
    float* const outs[4] = {out_albedo, out_normal, out_depth, out_coverage};
    const size_t n_pix = (size_t)P->width * P->height * n_frames, per[4] = {3, 3, 1, 1};
    size_t at[4], total = 0;
    float* first = nullptr;
    for (int k = 0; k < 4; ++k) {
        at[k] = total;
        total += outs[k] ? per[k] * n_pix : 0;
        if (!first) first = outs[k];
    }
    if (!first) return fail(c, VK_ERR_INVALID, who + ": every output is null");
    CU(c, cudaSetDevice(c->device));
    Staging S;
    if ((rc = stage(c, total, false, Outputs{first, nullptr, nullptr, nullptr, nullptr}, &S)) != VK_OK) return rc;
    float* dev[4];
    for (int k = 0; k < 4; ++k) dev[k] = outs[k] ? c->frame + at[k] : nullptr;
    RenderArgs a{};
    a.width = P->width;
    a.height = P->height;
    a.seed_lo = (uint32_t)P->seed;
    a.seed_hi = (uint32_t)(P->seed >> 32);
    a.background = make_float3(P->background[0], P->background[1], P->background[2]);
    a.flags = P->flags;
    a.tiles_x = (P->width + 7) / 8;
    a.tiles_y = (P->height + 3) / 4;
    const FlatProgram* flat = hit_program(c, P->flags);
    CU(c, cudaEventRecord(c->ev2, c->stream));
    CU(c, cudaEventRecord(c->ev0, c->stream));
    if ((rc = upload_cams(c, cams, n_frames)) != VK_OK) return rc;
    CU(c, (P->flags & VK_FLAG_STRICT_MATH ? vkstrict::launch_aov : vkfast::launch_aov)(c->scene, c->flat, flat != nullptr, c->cams, n_frames, a, aov_spp,
                                                                                     dev[0], dev[1], dev[2], dev[3], c->counters, c->stream));
    CU(c, cudaEventRecord(c->ev1, c->stream));
    c->launches += 1;
    c->paths += n_pix * aov_spp;
    vk_stats st{};
    if ((rc = vk_flush_stats(c, &st)) != VK_OK) return rc;
    CU(c, cudaEventElapsedTime(&st.ms_kernels, c->ev0, c->ev1));
    st.variant = VK_VARIANT_AUTO;
    size_t off[VK_CHUNKS + 1];
    if ((rc = chunks_begin(c, total, sizeof(float), off)) != VK_OK) return rc;
    CU(c, cudaEventRecord(c->ev1, c->stream));
    HostSpan spans[4];
    int n_spans = 0;
    for (int k = 0; k < 4; ++k)
        if (outs[k]) spans[n_spans++] = HostSpan{(char*)outs[k], at[k] * sizeof(float), (at[k] + per[k] * n_pix) * sizeof(float)};
    if ((rc = chunks_end(c, off, spans, n_spans)) != VK_OK) return rc;
    CU(c, cudaStreamSynchronize(c->stream));
    CU(c, cudaEventElapsedTime(&st.ms_total, c->ev2, c->ev1));
    if (stats) *stats = st;
    return VK_OK;
}

int vk_render_aov(vk_ctx* c, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P, uint32_t aov_spp, float* out_albedo,
                  float* out_normal, float* out_depth, float* out_coverage, vk_stats* stats) {
    return render_aov(c, "vk_render_aov", cams, n_frames, P, aov_spp, out_albedo, out_normal, out_depth, out_coverage, stats);
}

// ---- adaptive sessions (vk_adaptive_*; the one-shot vk_render_adaptive* calls run one on c->oneshot) ----
static void adaptive_free(vk_adaptive_session* s) {
    if (!s) return;
    if (s->block && s->c) {
        cudaSetDevice(s->c->device);
        cudaFree(s->block);
    }
    delete s;
}

// The pixels that render on from level l of a refine: those k_adaptive_levels marked with l + 1, in ascending order.
struct AtLevel {
    const uint32_t* level;
    uint32_t want;
    __device__ bool operator()(uint32_t p) const { return level[p] == want; }
};

// How many of n_pix pixels shard `shard` of n_shards owns (k_shard_list's rule): whole runs, less the missing tail of the
// last run when the shard owns it.
static uint32_t shard_pixels(uint32_t n_pix, uint32_t shard, uint32_t n_shards) {
    const uint32_t runs = (n_pix + VK_SHARD_RUN - 1) / VK_SHARD_RUN;
    if (runs <= shard) return 0u;
    const uint32_t owned_runs = (runs - 1u - shard) / n_shards + 1u;
    const uint32_t tail = (runs - 1u) % n_shards == shard ? runs * VK_SHARD_RUN - n_pix : 0u;
    return owned_runs * VK_SHARD_RUN - tail;
}

// Checks, plans the kernel, sizes s's buffers (a larger block than needed is reused) and zeroes its state.  The kernel is
// planned on the whole batch whatever the shard, so every shard runs the kernel the unsharded session runs.
static int adaptive_begin(vk_ctx* c, const std::string& w, const vk_camera* cam, uint32_t n_frames, const vk_render_params* P,
                          uint32_t pass_spp, float max_error, vk_adaptive_session* s, uint32_t shard = 0, uint32_t n_shards = 1) {
    s->c = c;
    int rc = check_render(c, w, cam, n_frames, P, true, pass_spp, max_error);
    if (rc != VK_OK) return rc;
    CU(c, cudaSetDevice(c->device));
    // AUTO decides once, on pass 0's path count; every pass of every refine runs that kernel
    vk_render_params Q = *P;
    Q.spp_count = pass_spp < P->spp ? pass_spp : P->spp;
    RenderPlan R;
    if ((rc = plan_render(c, w, &Q, n_frames, true, &R)) != VK_OK) return rc;

    const uint32_t n_pix = P->width * P->height * n_frames; // (all frames: a pixel index is batch-wide)
    const size_t plane = (size_t)n_pix * 3;
    const uint32_t max_levels = (P->spp - 1) / pass_spp + 1;
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    size_t sel_bytes = 0, lvl_bytes = 0;
    CU(c, cub::DeviceSelect::Flagged(nullptr, sel_bytes, (const uint32_t*)nullptr, (const uint8_t*)nullptr, (uint32_t*)nullptr, (int*)nullptr,
                                     (int)n_pix, c->stream));
    CU(c, cub::DeviceSelect::If(nullptr, lvl_bytes, thrust::counting_iterator<uint32_t>(0), (uint32_t*)nullptr, (int*)nullptr, (int)n_pix,
                                AtLevel{nullptr, 0}, c->stream));
    const size_t cub_bytes = sel_bytes > lvl_bytes ? sel_bytes : lvl_bytes;
    const size_t o_acc = 0, o_sq = o_acc + al(plane * 8), o_n = o_sq + al(plane * 8), o_l0 = o_n + al(n_pix * 4ull),
                 o_l1 = o_l0 + al(n_pix * 4ull), o_lv = o_l1 + al(n_pix * 4ull), o_nl = o_lv + al(n_pix * 4ull),
                 o_keep = o_nl + al(max_levels * 4ull), o_cnt = o_keep + al(n_pix), o_cub = o_cnt + 256, need = o_cub + al(cub_bytes);
    if (s->bytes < need) {
        if (s->block) cudaFree(s->block);
        s->block = nullptr;
        s->bytes = 0;
        CU(c, cudaMalloc(&s->block, need));
        s->bytes = need;
    }
    char* base = (char*)s->block;
    s->acc = (unsigned long long*)(base + o_acc);
    s->sq = (unsigned long long*)(base + o_sq);
    s->nspp = (uint32_t*)(base + o_n);
    s->cur = (uint32_t*)(base + o_l0);
    s->nxt = (uint32_t*)(base + o_l1);
    s->level = (uint32_t*)(base + o_lv);
    s->n_level = (uint32_t*)(base + o_nl);
    s->keep = (uint8_t*)(base + o_keep);
    s->d_count = (int*)(base + o_cnt);
    s->cub_tmp = base + o_cub;
    s->cub_bytes = cub_bytes;
    // a session starts with no samples: zero sums, squares and counts (the pass loop adds samples [n_p, ..) to them)
    CU(c, cudaMemsetAsync(base, 0, o_l0, c->stream));
    s->cams.assign(cam, cam + n_frames);
    s->P = *P;
    s->n_frames = n_frames;
    s->pass_spp = pass_spp;
    s->n_pix = n_pix;
    s->shard = shard;
    s->n_shards = n_shards;
    s->n_owned = shard_pixels(n_pix, shard, n_shards);
    s->max_levels = max_levels;
    s->R = R;
    s->scene_gen = c->scene_gen;
    s->reached_any = false;
    s->broken = false;
    s->reached = vk_adaptive_target{0, 0, 0.0f};
    return VK_OK;
}

// Whether T may follow what s has reached (include/vecchio_gpu.h, vk_adaptive_refine); a message when not.
static std::string adaptive_refusal(const vk_adaptive_session* s, const vk_adaptive_target& T) {
    if (T.spp == 0) return "the target's spp must be >= 1";
    if (T.spp > s->P.spp) return "the target's spp " + std::to_string(T.spp) + " exceeds the session's limit params->spp = " + std::to_string(s->P.spp);
    if (!(T.max_error >= 0.0f)) return "max_error must be >= 0 (and not NaN)";
    if (!s->reached_any) return "";
    const vk_adaptive_target& A = s->reached;
    if (A.max_error == 0.0f ? T.max_error != 0.0f : (T.max_error != 0.0f && T.max_error > A.max_error))
        return "max_error may only tighten (0 is the tightest: after 0 only 0 may follow)";
    if (T.min_spp < A.min_spp) return "min_spp may only rise";
    if (T.spp < A.spp) return "spp may only rise";
    if (T.spp > A.spp && A.spp % s->pass_spp != 0)
        return "spp may rise only from a cap on the pass grid (a multiple of pass_spp): pixels stopped at " + std::to_string(A.spp) +
               " would go on off the grid";
    return "";
}

// The pass loop of every adaptive render: renders s until target T is reached (the caller has checked T).  A fresh state is
// today's one-shot render: every pixel from level 0.  Otherwise k_adaptive_levels re-applies the rule of T to every pixel
// and counts per level those that render on; from the lowest non-empty level upward, each pass covers the pixels reopened
// at that level plus the survivors of the level below, and empty levels cost nothing.  Adds what it launched and the samples
// it started to *launches / *paths and the passes' kernel time to *ms_kernels.
static int adaptive_refine(vk_adaptive_session* s, const vk_adaptive_target& T, uint32_t* launches, uint64_t* paths, float* ms_kernels) {
    vk_ctx* c = s->c;
    const uint32_t M = s->pass_spp, n_pix = s->n_pix;
    CU(c, cudaSetDevice(c->device));
    int rc = ensure_pinned(c, (size_t)s->max_levels + 1);
    if (rc != VK_OK) return rc;
    uint32_t* h_count = (uint32_t*)c->pinned;
    uint32_t* h_level = h_count + 1;
    s->broken = true; // until the loop has run to its end
    const bool fresh = !s->reached_any;
    const uint32_t n_levels = (T.spp - 1) / M + 1; // levels 0 .. n_levels-1: pixels at l * M samples
    uint32_t *cur = s->cur, *nxt = s->nxt;
    // the list of level l's reopened pixels into `out` (their count is h_level[l])
    auto level_list = [&](uint32_t l, uint32_t* out) -> int {
        size_t bytes = s->cub_bytes;
        CU(c, cub::DeviceSelect::If(s->cub_tmp, bytes, thrust::counting_iterator<uint32_t>(0), out, s->d_count, (int)n_pix,
                                    AtLevel{s->level, l + 1u}, c->stream));
        *launches += 2; // (its init and select kernels)
        return VK_OK;
    };
    uint32_t lvl = 0, n_active = 0;
    if (s->n_owned == 0) { // a shard without pixels: nothing to render, and the target is reached
    } else if (fresh) {
        n_active = s->n_owned; // every owned pixel from level 0, ascending
        k_shard_list<<<(n_active + 255) / 256, 256, 0, c->stream>>>(cur, n_active, s->shard, s->n_shards);
        *launches += 1;
    } else {
        CU(c, cudaMemsetAsync(s->n_level, 0, n_levels * sizeof(uint32_t), c->stream));
        k_adaptive_levels<<<(n_pix + 255) / 256, 256, 0, c->stream>>>(s->acc, s->sq, s->nspp, n_pix, T.spp, T.min_spp, T.max_error, M,
                                                                      s->shard, s->n_shards, s->level, s->n_level);
        *launches += 1;
        CU(c, cudaGetLastError());
        CU(c, cudaMemcpyAsync(h_level, s->n_level, n_levels * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream)); // one read-back per refine: which levels have pixels
        while (lvl < n_levels && h_level[lvl] == 0u) ++lvl;
        if (lvl < n_levels) {
            if ((rc = level_list(lvl, cur)) != VK_OK) return rc;
            n_active = h_level[lvl];
        }
    }
    apply_l2_window(c);
    RenderBuffers b{};
    b.counters = c->counters;
    b.debug = c->debug;
    b.acc = s->acc;
    b.accsq = nullptr;
    while (n_active) {
        const uint32_t done = lvl * M, cnt = T.spp - done < M ? T.spp - done : M;
        const ListArgs la{cur, n_active, s->sq};
        CU(c, cudaEventRecord(c->ev0, c->stream));
        if ((rc = launch_pass(c, s->R, s->cams.data(), &s->P, done, cnt, b, s->n_frames, &la, launches)) != VK_OK) return rc;
        *paths += (uint64_t)n_active * cnt;
        k_adaptive_select<<<(n_active + 255) / 256, 256, 0, c->stream>>>(cur, n_active, s->acc, s->sq, done + cnt, T.spp, T.min_spp,
                                                                         T.max_error, s->nspp, s->keep);
        ++*launches;
        const bool last = done + cnt == T.spp;
        // the next list: level lvl + 1's reopened pixels, then the kept entries, compacted in their (ascending) order
        const uint32_t reopened = !fresh && lvl + 1 < n_levels ? h_level[lvl + 1] : 0u;
        if (!last) {
            if (reopened && (rc = level_list(lvl + 1, nxt)) != VK_OK) return rc;
            CU(c, cub::DeviceSelect::Flagged(s->cub_tmp, s->cub_bytes, cur, s->keep, nxt + reopened, s->d_count, (int)n_active, c->stream));
            *launches += 2;
        }
        CU(c, cudaGetLastError());
        CU(c, cudaEventRecord(c->ev1, c->stream));
        // one 4-byte D2H and a stream synchronisation per pass: the host sizes the next pass's work from the count
        if (!last) CU(c, cudaMemcpyAsync(h_count, s->d_count, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        float ms = 0.0f;
        CU(c, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
        *ms_kernels += ms;
        if (last) break;
        n_active = *h_count + reopened;
        ++lvl;
        std::swap(cur, nxt);
        if (n_active == 0 && !fresh) { // nothing left at this level: on to the next level with reopened pixels
            ++lvl;
            while (lvl < n_levels && h_level[lvl] == 0u) ++lvl;
            if (lvl < n_levels) {
                if ((rc = level_list(lvl, cur)) != VK_OK) return rc;
                n_active = h_level[lvl];
            }
        }
    }
    s->reached = T;
    s->reached_any = true;
    s->broken = false;
    return VK_OK;
}

// shared body of vk_render_adaptive* and vk_render_frames_adaptive* (include/vecchio_gpu.h states the passes and the rule):
// begin, one refine to {spp, 0, max_error} and read, on the context's own session.
// n_frames > 1: cams points to n_frames cameras, every pass runs one launch over the active pixels of all frames (one list of
// batch-wide pixels, FrameListArgs) and the result is n_frames contiguous planes.
static int render_adaptive(vk_ctx* c, const std::string& who, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P, uint32_t pass_spp,
                           float max_error, float* out_rgb, uint8_t* out_rgb8, uint32_t* out_spp, vk_stats* stats) {
    if (!c) return VK_ERR_INVALID;
    if (!out_rgb && !out_rgb8) return fail(c, VK_ERR_INVALID, who + ": null argument");
    if (!c->oneshot) c->oneshot = new vk_adaptive_session;
    vk_adaptive_session* s = c->oneshot;
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaEventRecord(c->ev2, c->stream));
    int rc = adaptive_begin(c, who, cams, n_frames, P, pass_spp, max_error, s);
    if (rc != VK_OK) return rc;
    uint32_t launches = 0;
    uint64_t paths = 0;
    float ms_kernels = 0.0f;
    if ((rc = adaptive_refine(s, vk_adaptive_target{P->spp, 0u, max_error}, &launches, &paths, &ms_kernels)) != VK_OK) return rc;
    c->launches += launches;
    c->paths += paths;
    vk_stats st{};
    if ((rc = vk_flush_stats(c, &st)) != VK_OK) return rc;
    st.ms_kernels = ms_kernels;
    st.variant = s->R.variant;
    if ((rc = readout(c, P, n_frames, s, Outputs{out_rgb, out_rgb8, nullptr, out_spp, nullptr}, &st)) != VK_OK) return rc;
    if (stats) *stats = st;
    return VK_OK;
}

int vk_render_adaptive(vk_ctx* c, const vk_camera* cam, const vk_render_params* P, uint32_t pass_spp, float max_error, float* out_rgb,
                       uint32_t* out_spp, vk_stats* stats) {
    return render_adaptive(c, "vk_render_adaptive", cam, 1, P, pass_spp, max_error, out_rgb, nullptr, out_spp, stats);
}

int vk_render_adaptive_rgb8(vk_ctx* c, const vk_camera* cam, const vk_render_params* P, uint32_t pass_spp, float max_error,
                            uint8_t* out_rgb8, uint32_t* out_spp, vk_stats* stats) {
    return render_adaptive(c, "vk_render_adaptive_rgb8", cam, 1, P, pass_spp, max_error, nullptr, out_rgb8, out_spp, stats);
}

int vk_render_frames_adaptive(vk_ctx* c, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P, uint32_t pass_spp,
                              float max_error, float* out_rgb, uint32_t* out_spp, vk_stats* stats) {
    return render_adaptive(c, "vk_render_frames_adaptive", cams, n_frames, P, pass_spp, max_error, out_rgb, nullptr, out_spp, stats);
}

int vk_render_frames_adaptive_rgb8(vk_ctx* c, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P, uint32_t pass_spp,
                                   float max_error, uint8_t* out_rgb8, uint32_t* out_spp, vk_stats* stats) {
    return render_adaptive(c, "vk_render_frames_adaptive_rgb8", cams, n_frames, P, pass_spp, max_error, nullptr, out_rgb8, out_spp, stats);
}

// shared body of vk_adaptive_begin and vk_adaptive_begin_shard
static int begin_session(vk_ctx* c, const std::string& w, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P,
                         uint32_t pass_spp, uint32_t shard, uint32_t n_shards, vk_adaptive_session** out) {
    if (!c) return VK_ERR_INVALID;
    if (!out) return fail(c, VK_ERR_INVALID, w + ": null argument");
    *out = nullptr;
    if (n_shards == 0 || shard >= n_shards) return fail(c, VK_ERR_INVALID, w + ": shard must be < n_shards (and n_shards >= 1)");
    vk_adaptive_session* s = new vk_adaptive_session;
    s->c = c;
    const int rc = adaptive_begin(c, w, cams, n_frames, P, pass_spp, 0.0f, s, shard, n_shards);
    if (rc != VK_OK) {
        adaptive_free(s);
        return rc;
    }
    *out = s;
    return VK_OK;
}

int vk_adaptive_begin(vk_ctx* c, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P, uint32_t pass_spp,
                      vk_adaptive_session** out) {
    return begin_session(c, "vk_adaptive_begin", cams, n_frames, P, pass_spp, 0, 1, out);
}

int vk_adaptive_begin_shard(vk_ctx* c, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P, uint32_t pass_spp,
                            uint32_t shard, uint32_t n_shards, vk_adaptive_session** out) {
    return begin_session(c, "vk_adaptive_begin_shard", cams, n_frames, P, pass_spp, shard, n_shards, out);
}

int vk_adaptive_refine(vk_adaptive_session* s, const vk_adaptive_target* T, vk_stats* stats) {
    if (!s) return VK_ERR_INVALID;
    vk_ctx* c = s->c;
    if (!T) return fail(c, VK_ERR_INVALID, "vk_adaptive_refine: null target");
    if (s->broken) return fail(c, VK_ERR_INVALID, "vk_adaptive_refine: an earlier refine or import failed part way; the session's state is lost");
    if (!c->has_scene || c->scene_gen != s->scene_gen)
        return fail(c, VK_ERR_INVALID, "vk_adaptive_refine: the scene changed since the session began");
    const std::string why = adaptive_refusal(s, *T);
    if (!why.empty()) return fail(c, VK_ERR_INVALID, "vk_adaptive_refine: " + why);
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaEventRecord(c->ev2, c->stream));
    uint32_t launches = 0;
    uint64_t paths = 0;
    float ms_kernels = 0.0f;
    int rc = adaptive_refine(s, *T, &launches, &paths, &ms_kernels);
    if (rc != VK_OK) return rc;
    CU(c, cudaEventRecord(c->ev1, c->stream));
    c->launches += launches;
    c->paths += paths;
    vk_stats st{};
    if ((rc = vk_flush_stats(c, &st)) != VK_OK) return rc;
    st.ms_kernels = ms_kernels;
    CU(c, cudaEventElapsedTime(&st.ms_total, c->ev2, c->ev1));
    st.variant = s->R.variant;
    if (stats) *stats = st;
    return VK_OK;
}

static int adaptive_read_call(vk_adaptive_session* s, const char* who, float* out_rgb, uint8_t* out_rgb8, uint32_t* out_spp, float* out_error) {
    if (!s) return VK_ERR_INVALID;
    vk_ctx* c = s->c;
    if (!out_rgb && !out_rgb8) return fail(c, VK_ERR_INVALID, std::string(who) + ": null argument");
    if (s->broken) return fail(c, VK_ERR_INVALID, std::string(who) + ": an earlier refine or import failed part way; the session's state is lost");
    return readout(c, &s->P, s->n_frames, s, Outputs{out_rgb, out_rgb8, nullptr, out_spp, out_error}, nullptr); // (no refine's stats)
}

int vk_adaptive_read(vk_adaptive_session* s, float* out_rgb, uint32_t* out_spp, float* out_error) {
    return adaptive_read_call(s, "vk_adaptive_read", out_rgb, nullptr, out_spp, out_error);
}

int vk_adaptive_read_rgb8(vk_adaptive_session* s, uint8_t* out_rgb8, uint32_t* out_spp, float* out_error) {
    return adaptive_read_call(s, "vk_adaptive_read_rgb8", nullptr, out_rgb8, out_spp, out_error);
}

// The state into host arrays (vk_adaptive_export's layout).
static int adaptive_export(vk_adaptive_session* s, int64_t* sums, uint64_t* squares, uint32_t* counts, vk_adaptive_target* reached) {
    vk_ctx* c = s->c;
    const size_t n_pix = s->n_pix;
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaMemcpyAsync(sums, s->acc, n_pix * 3 * sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(squares, s->sq, n_pix * 3 * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(counts, s->nspp, n_pix * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (reached) *reached = s->reached;
    return VK_OK;
}

int vk_adaptive_export(vk_adaptive_session* s, int64_t* sums, uint64_t* squares, uint32_t* counts, vk_adaptive_target* reached) {
    if (!s) return VK_ERR_INVALID;
    vk_ctx* c = s->c;
    if (!sums || !squares || !counts) return fail(c, VK_ERR_INVALID, "vk_adaptive_export: null argument");
    if (s->broken) return fail(c, VK_ERR_INVALID, "vk_adaptive_export: an earlier refine or import failed part way; the session's state is lost");
    return adaptive_export(s, sums, squares, counts, reached);
}

// What vk_adaptive_import refuses of a state for s (`w` prefixes the message); VK_OK when s may take it.
static int adaptive_import_check(vk_adaptive_session* s, const std::string& w, const int64_t* sums, const uint64_t* squares,
                                 const uint32_t* counts, const vk_adaptive_target& A) {
    vk_ctx* c = s->c;
    if (A.spp > s->P.spp) return fail(c, VK_ERR_INVALID, w + "the reached spp exceeds the session's limit params->spp");
    if (!(A.max_error >= 0.0f)) return fail(c, VK_ERR_INVALID, w + "the reached max_error must be >= 0 (and not NaN)");
    if (A.spp == 0 && (A.min_spp != 0 || A.max_error != 0.0f)) return fail(c, VK_ERR_INVALID, w + "a state that reached no target has spp, min_spp and max_error 0");
    for (size_t p = 0; p < s->n_pix; ++p) {
        const uint32_t n = counts[p];
        const bool nonzero = (sums[3 * p] | sums[3 * p + 1] | sums[3 * p + 2] | (int64_t)(squares[3 * p] | squares[3 * p + 1] | squares[3 * p + 2])) != 0;
        if (s->n_shards > 1 && (p / VK_SHARD_RUN) % s->n_shards != s->shard && (n != 0 || nonzero))
            return fail(c, VK_ERR_INVALID, w + "pixel " + std::to_string(p) + " is not this shard's but has samples or non-zero sums");
        if (n > A.spp) return fail(c, VK_ERR_INVALID, w + "pixel " + std::to_string(p) + " has more samples than the reached spp");
        if (n % s->pass_spp != 0 && n != A.spp)
            return fail(c, VK_ERR_INVALID, w + "pixel " + std::to_string(p) + " has a count off the pass grid (neither a multiple of pass_spp nor the reached spp)");
        if (n == 0 && nonzero)
            return fail(c, VK_ERR_INVALID, w + "pixel " + std::to_string(p) + " has no samples but non-zero sums");
    }
    return VK_OK;
}

// Replaces s's state by the checked arrays.
static int adaptive_import(vk_adaptive_session* s, const int64_t* sums, const uint64_t* squares, const uint32_t* counts,
                           const vk_adaptive_target& A) {
    vk_ctx* c = s->c;
    const size_t n_pix = s->n_pix;
    CU(c, cudaSetDevice(c->device));
    s->broken = true; // until every array has arrived
    CU(c, cudaMemcpyAsync(s->acc, sums, n_pix * 3 * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaMemcpyAsync(s->sq, squares, n_pix * 3 * sizeof(uint64_t), cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaMemcpyAsync(s->nspp, counts, n_pix * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    s->reached = A;
    s->reached_any = A.spp != 0;
    s->broken = false;
    return VK_OK;
}

int vk_adaptive_import(vk_adaptive_session* s, const int64_t* sums, const uint64_t* squares, const uint32_t* counts,
                       const vk_adaptive_target* reached) {
    if (!s) return VK_ERR_INVALID;
    if (!sums || !squares || !counts || !reached) return fail(s->c, VK_ERR_INVALID, "vk_adaptive_import: null argument");
    const int rc = adaptive_import_check(s, "vk_adaptive_import: ", sums, squares, counts, *reached);
    return rc != VK_OK ? rc : adaptive_import(s, sums, squares, counts, *reached);
}

uint32_t vk_adaptive_variant(const vk_adaptive_session* s) { return s ? s->R.variant : 0u; }

void vk_adaptive_destroy(vk_adaptive_session* s) { adaptive_free(s); }

int vk_intersect(vk_ctx* c, const vk_ray* rays, size_t n, const float* medium_xi, uint32_t flags, vk_hit* out) {
    if (!c) return VK_ERR_INVALID;
    if (!c->has_scene) return fail(c, VK_ERR_NO_SCENE, "vk_intersect: no scene uploaded");
    if (n == 0) return VK_OK;
    if (!rays || !out) return fail(c, VK_ERR_INVALID, "vk_intersect: null argument");
    if (medium_xi && c->n_media > VK_MEDIUM_XI_SLOTS / 2)
        return fail(c, VK_ERR_UNSUPPORTED, "vk_intersect: the injected variate table holds VK_MEDIUM_XI_SLOTS / 2 media (two visits each); this scene has more");
    CU(c, cudaSetDevice(c->device));
    vk_ray* d_rays = nullptr;
    vk_hit* d_hits = nullptr;
    float* d_xi = nullptr;
    int rc = VK_OK;
    cudaError_t e;
#define STEP(call)                                                                                                     \
    if (rc == VK_OK && (e = (call)) != cudaSuccess) rc = fail(c, VK_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e));
    STEP(cudaMalloc((void**)&d_rays, n * sizeof(vk_ray)))
    STEP(cudaMalloc((void**)&d_hits, n * sizeof(vk_hit)))
    if (medium_xi) {
        STEP(cudaMalloc((void**)&d_xi, n * VK_MEDIUM_XI_SLOTS * sizeof(float)))
        STEP(cudaMemcpyAsync(d_xi, medium_xi, n * VK_MEDIUM_XI_SLOTS * sizeof(float), cudaMemcpyHostToDevice, c->stream))
    }
    STEP(cudaMemcpyAsync(d_rays, rays, n * sizeof(vk_ray), cudaMemcpyHostToDevice, c->stream))
    const FlatProgram* flat = hit_program(c, flags);
    STEP((flags & VK_FLAG_STRICT_MATH) ? vkstrict::launch_intersect(c->scene, flat, d_rays, n, d_xi, d_hits, c->stream)
                                       : vkfast::launch_intersect(c->scene, flat, d_rays, n, d_xi, d_hits, c->stream))
    STEP(cudaMemcpyAsync(out, d_hits, n * sizeof(vk_hit), cudaMemcpyDeviceToHost, c->stream))
    STEP(cudaStreamSynchronize(c->stream))
#undef STEP
    cudaFree(d_rays);
    cudaFree(d_hits);
    cudaFree(d_xi);
    return rc;
}

// ------------------------------------------------------------------------------------------------
// One context over several GPUs of a node (SURVEY 8e): the frame's samples are split by global sample
// index, device k renders [k * spp / N, (k + 1) * spp / N) of every pixel into ITS integer accumulators,
// and device 0 adds the accumulators of its peers to its own by reading them over NVLink (peer-mapped
// loads from a reduce kernel: no staging copies, no host round trip, no communicator).  Integer sums:
// the frame is bit-identical to the one a single GPU renders for the same seed.
// ------------------------------------------------------------------------------------------------
#define VK_MULTI_MAX 16
struct PeerAcc {
    const unsigned long long* acc[VK_MULTI_MAX];
    const double* accsq[VK_MULTI_MAX];
    int n;
};
__global__ void k_reduce_peers(PeerAcc pa, size_t n, float* __restrict__ sum, float* __restrict__ sumsq) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    long long a = 0;
    for (int k = 0; k < pa.n; ++k) a += (long long)pa.acc[k][i]; // device 0's own buffer first, then the peers' (NVLink loads)
    sum[i] = (float)((double)a * VK_ACC_INV_SCALE);
    if (sumsq) {
        double q = 0.0;
        for (int k = 0; k < pa.n; ++k) q += pa.accsq[k][i];
        sumsq[i] = (float)q;
    }
}
// An adaptive session over the devices of a vk_multi (vk_multi_adaptive_*): device k holds shard k of n, an ordinary
// shard session (vk_adaptive_begin_shard's pixels) whose pass loop runs on its own thread during a refine.  A read or an
// export first gathers the owners' states into `comp`, an unsharded session's buffers on device 0, and then runs the
// single-context code on it.
struct vk_multi_adaptive_session {
    vk_multi* m = nullptr;
    std::vector<vk_adaptive_session*> shard; // shard k on device k
    vk_adaptive_session* comp = nullptr;     // device 0: the whole state, gathered from the shards
    bool comp_current = false;               // comp holds the shards' present state
    bool broken = false;                     // a refine or import failed part way on some shard: the state is lost
};
static void multi_adaptive_free(vk_multi_adaptive_session* ms) {
    if (!ms) return;
    for (vk_adaptive_session* s : ms->shard) adaptive_free(s);
    adaptive_free(ms->comp);
    delete ms;
}
// every pixel's sums, squares and count from the shard that owns it; the shards of devices 1.. are read over NVLink
// (vk_multi_create maps their memory on device 0)
struct ShardState {
    const unsigned long long* acc[VK_MULTI_MAX];
    const unsigned long long* sq[VK_MULTI_MAX];
    const uint32_t* nspp[VK_MULTI_MAX];
    uint32_t n;
};
__global__ void k_gather_shards(ShardState st, uint32_t n_pix, unsigned long long* __restrict__ acc, unsigned long long* __restrict__ sq,
                                uint32_t* __restrict__ nspp) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pix) return;
    const uint32_t k = (i / VK_SHARD_RUN) % st.n;
    for (uint32_t ch = 0; ch < 3u; ++ch) {
        acc[3u * i + ch] = st.acc[k][3u * i + ch];
        sq[3u * i + ch] = st.sq[k][3u * i + ch];
    }
    nspp[i] = st.nspp[k][i];
}

struct vk_multi {
    std::vector<vk_ctx*> ctx;
    std::vector<cudaEvent_t> done; // device k's slice has finished (recorded on its stream)
    std::string err;
    vk_multi_adaptive_session* oneshot = nullptr; // vk_multi_render_*adaptive_rgb8: the session each call begins, refines and reads
};
static thread_local std::string g_multi_err;
static int mfail(vk_multi* m, int code, const std::string& msg) {
    if (m) m->err = msg;
    else g_multi_err = msg;
    return code;
}

int vk_multi_create(const int* devices, int n, vk_multi** out) {
    if (!out) return mfail(nullptr, VK_ERR_INVALID, "vk_multi_create: null out pointer");
    *out = nullptr;
    if (!devices || n < 1 || n > VK_MULTI_MAX) return mfail(nullptr, VK_ERR_INVALID, "vk_multi_create: 1 .. 16 devices");
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < i; ++j)
            if (devices[i] == devices[j]) return mfail(nullptr, VK_ERR_INVALID, "vk_multi_create: a device is listed twice");
    vk_multi* m = new vk_multi;
    for (int i = 0; i < n; ++i) {
        vk_ctx* c = nullptr;
        const int rc = vk_create(devices[i], &c);
        if (rc != VK_OK) {
            g_multi_err = std::string("vk_multi_create: ") + vk_last_error(nullptr);
            vk_multi_destroy(m);
            return rc;
        }
        m->ctx.push_back(c);
        cudaEvent_t ev = nullptr;
        cudaSetDevice(devices[i]);
        cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
        m->done.push_back(ev);
    }
    // device 0 reads every peer's accumulators
    cudaSetDevice(devices[0]);
    for (int i = 1; i < n; ++i) {
        int can = 0;
        cudaDeviceCanAccessPeer(&can, devices[0], devices[i]);
        if (!can) {
            g_multi_err = "vk_multi_create: device " + std::to_string(devices[0]) + " cannot map the memory of device " + std::to_string(devices[i]) +
                          " (no peer access); there is no staged fallback";
            vk_multi_destroy(m);
            return VK_ERR_UNSUPPORTED;
        }
        const cudaError_t e = cudaDeviceEnablePeerAccess(devices[i], 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
            g_multi_err = std::string("vk_multi_create: cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e);
            vk_multi_destroy(m);
            return VK_ERR_CUDA;
        }
        cudaGetLastError();
    }
    *out = m;
    return VK_OK;
}
void vk_multi_destroy(vk_multi* m) {
    if (!m) return;
    multi_adaptive_free(m->oneshot);
    for (size_t i = 0; i < m->ctx.size(); ++i) {
        if (i < m->done.size() && m->done[i]) {
            cudaSetDevice(m->ctx[i]->device);
            cudaEventDestroy(m->done[i]);
        }
        vk_destroy(m->ctx[i]);
    }
    delete m;
}
const char* vk_multi_last_error(const vk_multi* m) { return m ? m->err.c_str() : g_multi_err.c_str(); }
int vk_multi_device_count(const vk_multi* m) { return m ? (int)m->ctx.size() : 0; }

int vk_multi_scene_upload(vk_multi* m, const vk_scene_desc* scene) {
    if (!m) return VK_ERR_INVALID;
    for (vk_ctx* c : m->ctx) {
        const int rc = vk_scene_upload(c, scene);
        if (rc != VK_OK) return mfail(m, rc, c->err);
    }
    return VK_OK;
}

// a CUDA call made for a vk_multi: its error is the vk_multi's
#define CUM(m, call)                                                                                                   \
    do {                                                                                                               \
        cudaError_t e_ = (call);                                                                                       \
        if (e_ != cudaSuccess)                                                                                         \
            return mfail(m, e_ == cudaErrorMemoryAllocation ? VK_ERR_OOM : VK_ERR_CUDA,                                \
                         std::string(#call) + ": " + cudaGetErrorString(e_));                                          \
    } while (0)

// shared body of vk_multi_render, vk_multi_render_rgb8 and vk_multi_render_frames_rgb8: every device accumulates its sample
// slice of every frame, device 0 adds the slices up into its staging (k_reduce_peers) and runs the readout
static int multi_render(vk_multi* m, const std::string& who, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P, float* out_rgb,
                        uint8_t* out_rgb8, float* out_sumsq, vk_stats* stats) {
    if (!m) return VK_ERR_INVALID;
    if (!out_rgb && !out_rgb8) return mfail(m, VK_ERR_INVALID, who + ": null argument");
    for (vk_ctx* c : m->ctx) { // every device, before any of them launches
        const int rc = check_render(c, who, cams, n_frames, P);
        if (rc != VK_OK) return mfail(m, rc, c->err);
    }
    const int n = (int)m->ctx.size();
    const uint32_t begin = P->spp_begin, count = P->spp_count ? P->spp_count : P->spp - P->spp_begin;
    const size_t plane = (size_t)P->width * P->height * 3 * n_frames;
    const Outputs o{out_rgb, out_rgb8, out_sumsq, nullptr, nullptr};
    vk_ctx* c0 = m->ctx[0];
    CUM(m, cudaSetDevice(c0->device));
    Staging S;
    int rc = stage(c0, plane, true, o, &S);
    if (rc != VK_OK) return mfail(m, rc, c0->err);
    CUM(m, cudaEventRecord(c0->ev2, c0->stream));
    int active = 0;
    PeerAcc pa{};
    for (int k = 0; k < n; ++k) { // global samples [begin + k * count / n, begin + (k + 1) * count / n)
        const uint32_t s0 = begin + (uint32_t)((uint64_t)count * k / n), s1 = begin + (uint32_t)((uint64_t)count * (k + 1) / n);
        if (s1 == s0) continue; // more devices than samples
        vk_render_params q = *P;
        q.spp_begin = s0;
        q.spp_count = s1 - s0;
        vk_ctx* c = m->ctx[k];
        if ((rc = render_into(c, cams, &q, nullptr, nullptr, nullptr, true, out_sumsq != nullptr, n_frames)) != VK_OK) return mfail(m, rc, c->err);
        CUM(m, cudaSetDevice(c->device));
        CUM(m, cudaEventRecord(m->done[k], c->stream));
        pa.acc[active] = (const unsigned long long*)c->partial;
        pa.accsq[active] = out_sumsq ? (const double*)(c->partial + plane * 2) : nullptr;
        ++active;
    }
    // device 0's stream waits for every slice, then reads the peers' accumulators
    CUM(m, cudaSetDevice(c0->device));
    for (int k = 0; k < n; ++k) CUM(m, cudaStreamWaitEvent(c0->stream, m->done[k], 0));
    pa.n = active;
    k_reduce_peers<<<(unsigned)((plane + 255) / 256), 256, 0, c0->stream>>>(pa, plane, c0->frame + S.sum, out_sumsq ? c0->frame + S.sumsq : nullptr);
    CUM(m, cudaGetLastError());
    c0->launches += 1;
    // counters of all devices (synchronises each)
    vk_stats st{};
    float ms_max = 0.0f;
    for (int k = 0; k < n; ++k) {
        vk_stats s{};
        vk_ctx* c = m->ctx[k];
        if ((rc = vk_flush_stats(c, &s)) != VK_OK) return mfail(m, rc, c->err);
        float ms = 0.0f;
        if (s.paths) CUM(m, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
        ms_max = ms > ms_max ? ms : ms_max;
        st.paths += s.paths; st.rays += s.rays; st.dropped_samples += s.dropped_samples;
        st.node_visits += s.node_visits; st.prim_tests += s.prim_tests; st.launches += s.launches;
    }
    st.ms_kernels = ms_max; // the slowest device's render kernels
    st.variant = VK_VARIANT_AUTO;
    if ((rc = readout(c0, P, n_frames, nullptr, o, &st)) != VK_OK) return mfail(m, rc, c0->err);
    if (stats) *stats = st;
    return VK_OK;
}

int vk_multi_render(vk_multi* m, const vk_camera* cam, const vk_render_params* P, float* out_rgb, float* out_sumsq, vk_stats* stats) {
    return multi_render(m, "vk_multi_render", cam, 1, P, out_rgb, nullptr, out_sumsq, stats);
}

int vk_multi_render_rgb8(vk_multi* m, const vk_camera* cam, const vk_render_params* P, uint8_t* out_rgb8, vk_stats* stats) {
    return multi_render(m, "vk_multi_render_rgb8", cam, 1, P, nullptr, out_rgb8, nullptr, stats);
}

int vk_multi_render_frames_rgb8(vk_multi* m, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P, uint8_t* out_rgb8,
                                vk_stats* stats) {
    return multi_render(m, "vk_multi_render_frames_rgb8", cams, n_frames, P, nullptr, out_rgb8, nullptr, stats);
}

// the planes are small next to a render: device 0 computes them all, the bytes of a one-GPU call
int vk_multi_render_aov(vk_multi* m, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P, uint32_t aov_spp, float* out_albedo,
                        float* out_normal, float* out_depth, float* out_coverage, vk_stats* stats) {
    if (!m) return VK_ERR_INVALID;
    vk_ctx* c0 = m->ctx[0];
    const int rc = render_aov(c0, "vk_multi_render_aov", cams, n_frames, P, aov_spp, out_albedo, out_normal, out_depth, out_coverage, stats);
    return rc == VK_OK ? rc : mfail(m, rc, c0->err);
}

// ---- adaptive sessions over several GPUs (include/vecchio_gpu.h, vk_multi_adaptive_begin) ----
static const char* const k_multi_lost = ": an earlier refine or import failed part way; the session's state is lost";

// Checks and begins shard k of n on device k, and the composite on device 0, all with zero state.
static int multi_adaptive_begin(vk_multi* m, const std::string& w, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P,
                                uint32_t pass_spp, float max_error, vk_multi_adaptive_session* ms) {
    const uint32_t n = (uint32_t)m->ctx.size();
    ms->m = m;
    ms->shard.resize(n, nullptr);
    for (uint32_t k = 0; k < n; ++k) {
        if (!ms->shard[k]) ms->shard[k] = new vk_adaptive_session;
        const int rc = adaptive_begin(m->ctx[k], w, cams, n_frames, P, pass_spp, max_error, ms->shard[k], k, n);
        if (rc != VK_OK) return mfail(m, rc, m->ctx[k]->err);
    }
    if (!ms->comp) ms->comp = new vk_adaptive_session;
    const int rc = adaptive_begin(m->ctx[0], w, cams, n_frames, P, pass_spp, max_error, ms->comp);
    if (rc != VK_OK) return mfail(m, rc, m->ctx[0]->err);
    ms->comp_current = true; // (zero, like every shard)
    ms->broken = false;
    return VK_OK;
}

// Every shard's refine to T at once, one host thread per device (each pass of a shard ends in a host synchronisation of its
// device), all joined before the stats are summed: paths, rays, dropped samples and launches over all devices, ms_kernels
// the slowest device's.
static int multi_adaptive_refine(vk_multi_adaptive_session* ms, const std::string& w, const vk_adaptive_target& T, vk_stats* out) {
    vk_multi* m = ms->m;
    const size_t n = ms->shard.size();
    for (size_t k = 0; k < n; ++k) {
        vk_ctx* c = m->ctx[k];
        if (!c->has_scene || c->scene_gen != ms->shard[k]->scene_gen) return mfail(m, VK_ERR_INVALID, w + ": the scene changed since the session began");
    }
    const std::string why = adaptive_refusal(ms->shard[0], T);
    if (!why.empty()) return mfail(m, VK_ERR_INVALID, w + ": " + why);
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<int> rc(n, VK_OK);
    std::vector<uint32_t> launches(n, 0u);
    std::vector<uint64_t> paths(n, 0u);
    std::vector<float> ms_k(n, 0.0f);
    auto run = [&](size_t k) { rc[k] = adaptive_refine(ms->shard[k], T, &launches[k], &paths[k], &ms_k[k]); };
    ms->comp_current = false;
    ms->broken = true; // until every shard has reached T
    {
        std::vector<std::thread> threads;
        for (size_t k = 1; k < n; ++k) {
            try {
                threads.emplace_back(run, k);
            } catch (...) { // no thread to be had: this shard runs on the calling thread after shard 0
                threads.emplace_back();
            }
        }
        run(0);
        for (size_t k = 1; k < n; ++k) {
            if (threads[k - 1].joinable()) threads[k - 1].join();
            else run(k);
        }
    }
    vk_stats total{};
    for (size_t k = 0; k < n; ++k) {
        vk_ctx* c = m->ctx[k];
        if (rc[k] != VK_OK) return mfail(m, rc[k], w + ": device " + std::to_string(c->device) + ": " + c->err);
        c->launches += launches[k];
        c->paths += paths[k];
        vk_stats s{};
        const int r = vk_flush_stats(c, &s);
        if (r != VK_OK) return mfail(m, r, w + ": " + c->err);
        total.paths += s.paths; total.rays += s.rays; total.dropped_samples += s.dropped_samples;
        total.node_visits += s.node_visits; total.prim_tests += s.prim_tests; total.launches += s.launches;
        total.ms_kernels = ms_k[k] > total.ms_kernels ? ms_k[k] : total.ms_kernels;
    }
    total.ms_total = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    total.variant = ms->shard[0]->R.variant;
    ms->broken = false;
    if (out) *out = total;
    return VK_OK;
}

// The composite on device 0 after a refine: one launch of k_gather_shards (a read or an export synchronises device 0
// before it returns, so no shard is written while the gather reads it).
static int multi_adaptive_composite(vk_multi_adaptive_session* ms, const std::string& w) {
    if (ms->comp_current) return VK_OK;
    vk_multi* m = ms->m;
    vk_adaptive_session* cs = ms->comp;
    ShardState st{};
    st.n = (uint32_t)ms->shard.size();
    for (uint32_t k = 0; k < st.n; ++k) {
        st.acc[k] = ms->shard[k]->acc;
        st.sq[k] = ms->shard[k]->sq;
        st.nspp[k] = ms->shard[k]->nspp;
    }
    vk_ctx* c0 = m->ctx[0];
    cudaError_t e = cudaSetDevice(c0->device);
    if (e == cudaSuccess) {
        k_gather_shards<<<(cs->n_pix + 255) / 256, 256, 0, c0->stream>>>(st, cs->n_pix, cs->acc, cs->sq, cs->nspp);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return mfail(m, VK_ERR_CUDA, w + ": k_gather_shards: " + cudaGetErrorString(e));
    cs->reached = ms->shard[0]->reached;
    cs->reached_any = ms->shard[0]->reached_any;
    ms->comp_current = true;
    return VK_OK;
}

static int multi_adaptive_read_call(vk_multi_adaptive_session* ms, const std::string& w, float* out_rgb, uint8_t* out_rgb8, uint32_t* out_spp,
                                    float* out_error) {
    if (!ms) return VK_ERR_INVALID;
    vk_multi* m = ms->m;
    if (!out_rgb && !out_rgb8) return mfail(m, VK_ERR_INVALID, w + ": null argument");
    if (ms->broken) return mfail(m, VK_ERR_INVALID, w + k_multi_lost);
    int rc = multi_adaptive_composite(ms, w);
    if (rc != VK_OK) return rc;
    rc = readout(m->ctx[0], &ms->comp->P, ms->comp->n_frames, ms->comp, Outputs{out_rgb, out_rgb8, nullptr, out_spp, out_error}, nullptr);
    return rc == VK_OK ? VK_OK : mfail(m, rc, w + ": " + m->ctx[0]->err);
}

// shared body of vk_multi_render_adaptive_rgb8 and vk_multi_render_frames_adaptive_rgb8: begin, one refine to
// {spp, 0, max_error} and read, on the vk_multi's own session
static int multi_render_adaptive(vk_multi* m, const std::string& w, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P,
                                 uint32_t pass_spp, float max_error, uint8_t* out_rgb8, uint32_t* out_spp, vk_stats* stats) {
    if (!m) return VK_ERR_INVALID;
    if (!out_rgb8) return mfail(m, VK_ERR_INVALID, w + ": null argument");
    const auto t0 = std::chrono::steady_clock::now();
    if (!m->oneshot) m->oneshot = new vk_multi_adaptive_session;
    vk_multi_adaptive_session* ms = m->oneshot;
    int rc = multi_adaptive_begin(m, w, cams, n_frames, P, pass_spp, max_error, ms);
    if (rc != VK_OK) return rc;
    vk_stats st{};
    if ((rc = multi_adaptive_refine(ms, w, vk_adaptive_target{P->spp, 0u, max_error}, &st)) != VK_OK) return rc;
    if ((rc = multi_adaptive_read_call(ms, w, nullptr, out_rgb8, out_spp, nullptr)) != VK_OK) return rc;
    st.launches += 2; // (the gather and the readout)
    st.ms_total = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats) *stats = st;
    return VK_OK;
}

int vk_multi_render_adaptive_rgb8(vk_multi* m, const vk_camera* cam, const vk_render_params* P, uint32_t pass_spp, float max_error,
                                  uint8_t* out_rgb8, uint32_t* out_spp, vk_stats* stats) {
    return multi_render_adaptive(m, "vk_multi_render_adaptive_rgb8", cam, 1, P, pass_spp, max_error, out_rgb8, out_spp, stats);
}

int vk_multi_render_frames_adaptive_rgb8(vk_multi* m, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P, uint32_t pass_spp,
                                         float max_error, uint8_t* out_rgb8, uint32_t* out_spp, vk_stats* stats) {
    return multi_render_adaptive(m, "vk_multi_render_frames_adaptive_rgb8", cams, n_frames, P, pass_spp, max_error, out_rgb8, out_spp, stats);
}

int vk_multi_adaptive_begin(vk_multi* m, const vk_camera* cams, uint32_t n_frames, const vk_render_params* P, uint32_t pass_spp,
                            vk_multi_adaptive_session** out) {
    if (!m) return VK_ERR_INVALID;
    if (!out) return mfail(m, VK_ERR_INVALID, "vk_multi_adaptive_begin: null argument");
    *out = nullptr;
    vk_multi_adaptive_session* ms = new vk_multi_adaptive_session;
    const int rc = multi_adaptive_begin(m, "vk_multi_adaptive_begin", cams, n_frames, P, pass_spp, 0.0f, ms);
    if (rc != VK_OK) {
        multi_adaptive_free(ms);
        return rc;
    }
    *out = ms;
    return VK_OK;
}

int vk_multi_adaptive_refine(vk_multi_adaptive_session* ms, const vk_adaptive_target* T, vk_stats* stats) {
    if (!ms) return VK_ERR_INVALID;
    if (!T) return mfail(ms->m, VK_ERR_INVALID, "vk_multi_adaptive_refine: null target");
    if (ms->broken) return mfail(ms->m, VK_ERR_INVALID, std::string("vk_multi_adaptive_refine") + k_multi_lost);
    return multi_adaptive_refine(ms, "vk_multi_adaptive_refine", *T, stats);
}

int vk_multi_adaptive_read(vk_multi_adaptive_session* ms, float* out_rgb, uint32_t* out_spp, float* out_error) {
    return multi_adaptive_read_call(ms, "vk_multi_adaptive_read", out_rgb, nullptr, out_spp, out_error);
}

int vk_multi_adaptive_read_rgb8(vk_multi_adaptive_session* ms, uint8_t* out_rgb8, uint32_t* out_spp, float* out_error) {
    return multi_adaptive_read_call(ms, "vk_multi_adaptive_read_rgb8", nullptr, out_rgb8, out_spp, out_error);
}

int vk_multi_adaptive_export(vk_multi_adaptive_session* ms, int64_t* sums, uint64_t* squares, uint32_t* counts, vk_adaptive_target* reached) {
    if (!ms) return VK_ERR_INVALID;
    vk_multi* m = ms->m;
    const std::string w = "vk_multi_adaptive_export";
    if (!sums || !squares || !counts) return mfail(m, VK_ERR_INVALID, w + ": null argument");
    if (ms->broken) return mfail(m, VK_ERR_INVALID, w + k_multi_lost);
    int rc = multi_adaptive_composite(ms, w);
    if (rc != VK_OK) return rc;
    rc = adaptive_export(ms->comp, sums, squares, counts, reached);
    return rc == VK_OK ? VK_OK : mfail(m, rc, w + ": " + m->ctx[0]->err);
}

// The whole state is checked as vk_adaptive_import checks it (which is what every shard's check of its part adds up to:
// the parts carry zeros on the pixels a shard does not own), then each shard takes its owned pixels and the composite
// takes the whole.
int vk_multi_adaptive_import(vk_multi_adaptive_session* ms, const int64_t* sums, const uint64_t* squares, const uint32_t* counts,
                             const vk_adaptive_target* reached) {
    if (!ms) return VK_ERR_INVALID;
    vk_multi* m = ms->m;
    const std::string w = "vk_multi_adaptive_import: ";
    if (!sums || !squares || !counts || !reached) return mfail(m, VK_ERR_INVALID, w + "null argument");
    vk_adaptive_session* cs = ms->comp;
    int rc = adaptive_import_check(cs, w, sums, squares, counts, *reached);
    if (rc != VK_OK) return mfail(m, rc, m->ctx[0]->err);
    const size_t n_pix = cs->n_pix, n = ms->shard.size();
    ms->broken = true; // until every shard has its part
    ms->comp_current = false;
    std::vector<int64_t> s_part(n_pix * 3);
    std::vector<uint64_t> q_part(n_pix * 3);
    std::vector<uint32_t> n_part(n_pix);
    for (size_t k = 0; k < n; ++k) {
        for (size_t p = 0; p < n_pix; ++p) {
            const bool own = (p / VK_SHARD_RUN) % n == k;
            for (size_t ch = 0; ch < 3; ++ch) {
                s_part[3 * p + ch] = own ? sums[3 * p + ch] : 0;
                q_part[3 * p + ch] = own ? squares[3 * p + ch] : 0u;
            }
            n_part[p] = own ? counts[p] : 0u;
        }
        if ((rc = adaptive_import(ms->shard[k], s_part.data(), q_part.data(), n_part.data(), *reached)) != VK_OK)
            return mfail(m, rc, w + m->ctx[k]->err);
    }
    if ((rc = adaptive_import(cs, sums, squares, counts, *reached)) != VK_OK) return mfail(m, rc, w + m->ctx[0]->err);
    ms->comp_current = true;
    ms->broken = false;
    return VK_OK;
}

uint32_t vk_multi_adaptive_variant(const vk_multi_adaptive_session* ms) { return ms && !ms->shard.empty() ? ms->shard[0]->R.variant : 0u; }

void vk_multi_adaptive_destroy(vk_multi_adaptive_session* ms) { multi_adaptive_free(ms); }

int vk_eval_batch(vk_ctx* c, vk_eval* recs, size_t n, uint32_t flags) {
    if (!c) return VK_ERR_INVALID;
    if (!c->has_scene) return fail(c, VK_ERR_NO_SCENE, "vk_eval_batch: no scene uploaded");
    if (n == 0) return VK_OK;
    if (!recs) return fail(c, VK_ERR_INVALID, "vk_eval_batch: null argument");
    for (size_t i = 0; i < n; ++i) {
        const vk_eval& e = recs[i];
        const bool bounce = e.op == VK_EVAL_BOUNCE || e.op == VK_EVAL_BOUNCE_LEGACY;
        if (e.op > VK_EVAL_LIGHT_RANDOM || (bounce && e.index >= c->n_materials) || (e.op == VK_EVAL_TEXTURE && e.index >= c->n_textures) ||
            (e.op == VK_EVAL_LIGHT_RANDOM && e.index >= c->scene.n_lights))
            return fail(c, VK_ERR_INVALID, "vk_eval_batch: record " + std::to_string(i) + ": bad op or index");
        if (e.op == VK_EVAL_BOUNCE_LEGACY && c->has_specdiffuse)
            return fail(c, VK_ERR_UNSUPPORTED, "vk_eval_batch: SpecDiffuse has no legacy scatter (src/material.rs:21-28)");
        if ((e.op == VK_EVAL_BOUNCE || e.op == VK_EVAL_LIGHTS_PDF) && c->scene.n_lights == 0)
            return fail(c, VK_ERR_INVALID, "vk_eval_batch: empty light list (the reference panics, src/hittable.rs:431)");
    }
    CU(c, cudaSetDevice(c->device));
    vk_eval* d = nullptr;
    int rc = VK_OK;
    cudaError_t e;
#define STEP(call)                                                                                                     \
    if (rc == VK_OK && (e = (call)) != cudaSuccess) rc = fail(c, VK_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e));
    STEP(cudaMalloc((void**)&d, n * sizeof(vk_eval)))
    STEP(cudaMemcpyAsync(d, recs, n * sizeof(vk_eval), cudaMemcpyHostToDevice, c->stream))
    STEP((flags & VK_FLAG_STRICT_MATH) ? vkstrict::launch_eval(c->scene, d, n, c->n_materials, c->n_textures, c->stream)
                                       : vkfast::launch_eval(c->scene, d, n, c->n_materials, c->n_textures, c->stream))
    STEP(cudaMemcpyAsync(recs, d, n * sizeof(vk_eval), cudaMemcpyDeviceToHost, c->stream))
    STEP(cudaStreamSynchronize(c->stream))
#undef STEP
    cudaFree(d);
    return rc;
}

int vk_measure_peaks(vk_ctx* c, float* fp32_tflops, float* l2_gbs) {
    if (!c) return VK_ERR_INVALID;
    CU(c, cudaSetDevice(c->device));
    float* out = nullptr;
    const int blocks = c->sm_count * 8, threads = 256, iters = 4096;
    CU(c, cudaMalloc((void**)&out, (size_t)blocks * threads * sizeof(float)));
    float best_ms = 1e30f, ms = 0.f;
    for (int r = 0; r < 5; ++r) {
        cudaEventRecord(c->ev0, c->stream);
        k_ffma_peak<<<blocks, threads, 0, c->stream>>>(out, iters);
        cudaEventRecord(c->ev1, c->stream);
        cudaStreamSynchronize(c->stream);
        cudaEventElapsedTime(&ms, c->ev0, c->ev1);
        if (r > 0 && ms < best_ms) best_ms = ms;
    }
    if (fp32_tflops) *fp32_tflops = (float)((double)blocks * threads * iters * 16.0 * 8.0 * 2.0 / (best_ms * 1e-3) / 1e12);
    cudaFree(out);
    const size_t bytes = 32ull << 20; // 32 MiB: well inside the 126 MB L2
    float4* buf = nullptr;
    float* sink = nullptr;
    CU(c, cudaMalloc((void**)&buf, bytes));
    CU(c, cudaMalloc((void**)&sink, sizeof(float)));
    CU(c, cudaMemsetAsync(buf, 0, bytes, c->stream));
    const int reps = 20;
    best_ms = 1e30f;
    for (int r = 0; r < 5; ++r) {
        cudaEventRecord(c->ev0, c->stream);
        k_l2_read<<<c->sm_count * 8, 256, 0, c->stream>>>(buf, bytes / sizeof(float4), reps, sink);
        cudaEventRecord(c->ev1, c->stream);
        cudaStreamSynchronize(c->stream);
        cudaEventElapsedTime(&ms, c->ev0, c->ev1);
        if (r > 0 && ms < best_ms) best_ms = ms;
    }
    if (l2_gbs) *l2_gbs = (float)((double)bytes * reps / (best_ms * 1e-3) / 1e9);
    cudaFree(buf);
    cudaFree(sink);
    CU(c, cudaGetLastError());
    return VK_OK;
}

// Debug hook: the raw counter block (see RenderBuffers); [5..7] = first CTA start, first and last CTA end of the
// last staged launch (globaltimer ns).
int vk_debug_counters(vk_ctx* c, unsigned long long out[8]) {
    if (!c || !out) return VK_ERR_INVALID;
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaStreamSynchronize(c->stream));
    CU(c, cudaMemcpy(out, c->counters, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return VK_OK;
}
int vk_debug_ctas(vk_ctx* c, unsigned long long* out, size_t n_ctas) {
    if (!c || !out || n_ctas > VK_DEBUG_CTAS) return VK_ERR_INVALID;
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaStreamSynchronize(c->stream));
    CU(c, cudaMemcpy(out, c->debug, n_ctas * 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return VK_OK;
}

// Test hook: Philox4x32-10 on the device for the Random123 known-answer vectors.
int vk_selftest_philox(vk_ctx* c, const uint32_t ctr_key6[6], uint32_t out4[4]) {
    if (!c || !ctr_key6 || !out4) return VK_ERR_INVALID;
    CU(c, cudaSetDevice(c->device));
    uint32_t* d = nullptr;
    CU(c, cudaMalloc((void**)&d, 10 * sizeof(uint32_t)));
    cudaMemcpyAsync(d, ctr_key6, 6 * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream);
    cudaError_t e = vkfast::launch_philox_kat(d, d + 6, c->stream);
    cudaMemcpyAsync(out4, d + 6, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream);
    cudaStreamSynchronize(c->stream);
    cudaFree(d);
    CU(c, e);
    CU(c, cudaGetLastError());
    return VK_OK;
}

} // extern "C"
