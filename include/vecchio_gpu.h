/*
 * vecchio_gpu.h -- C ABI of the B200 (sm_100a) path-tracing sample loop.
 *
 * This is the drop-in boundary for the ONE hot path of browserdotsys/vecchio: the
 * per-pixel sample loop of the reference, `src/main.rs:181-198`, and everything it
 * calls (`ray_color` `src/main.rs:123-153`, every `Hittable::hit`, `Material::
 * scatter_with_pdf`, `Texture::value`, the PDF objects of `src/util.rs`).
 *
 * The reference has no FFI of its own (pure safe Rust).  The entry points below are
 * what a `gpu` module of the Rust host would bind with `extern "C"` (see
 * INTEGRATION.md and rust/gpu.rs); each one names the reference code it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; caller owns every host buffer; the library
 *     keeps no pointer after a call returns.
 *   - every function returns VK_OK (0) or a negative vk_status; the message is
 *     available from vk_last_error().  Nothing aborts or throws across the ABI.
 *   - there is NO CPU fallback: without a CUDA device vk_create fails with
 *     VK_ERR_NO_DEVICE, and a scene element the GPU path does not implement fails
 *     vk_scene_upload with VK_ERR_UNSUPPORTED.
 *   - all arithmetic is IEEE fp32, like the reference (`f32`, `src/vec3.rs:3-8`).
 */
#ifndef VECCHIO_GPU_H
#define VECCHIO_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VK_API_VERSION 1u

typedef enum vk_status {
    VK_OK = 0,
    VK_ERR_INVALID = -1,     /* bad argument / malformed scene description          */
    VK_ERR_NO_DEVICE = -2,   /* no CUDA device (there is no CPU fallback)           */
    VK_ERR_CUDA = -3,        /* a CUDA runtime call failed                          */
    VK_ERR_UNSUPPORTED = -4, /* scene element not implemented on the GPU path       */
    VK_ERR_NO_SCENE = -5,    /* render/intersect before vk_scene_upload             */
    VK_ERR_OOM = -6
} vk_status;

/* ------------------------------------------------------------------------------
 * Flattened scene.  The reference's object graph of `Arc<dyn Hittable>` trait
 * objects (`src/hittable.rs:33-44`) is lowered to one typed record array per
 * primitive kind plus 32-bit tagged references between them.
 * ---------------------------------------------------------------------------- */

typedef uint32_t vk_ref; /* (type << 28) | index ; 0 == none */

enum {
    VK_T_NONE = 0,
    VK_T_NODE = 1,    /* BVHNode            src/accel.rs:52-83                 */
    VK_T_SPHERE = 2,  /* Sphere             src/hittable.rs:46-121             */
    VK_T_MSPHERE = 3, /* MovingSphere       src/hittable.rs:136-197            */
    VK_T_RECT = 4,    /* Rect (+FlipFace)   src/hittable.rs:199-312            */
    VK_T_BOX = 5,     /* Boxy               src/hittable.rs:314-378            */
    VK_T_XFORM = 6,   /* Translate/Rotate{X,Y,Z}/FlipFace  :294-312, :500-807  */
    VK_T_MEDIUM = 7   /* ConstantMedium     src/hittable.rs:436-498            */
};
#define VK_REF_NONE 0u
#define VK_REF(type, index) ((((uint32_t)(type)) << 28) | ((uint32_t)(index) & 0x0FFFFFFFu))
#define VK_REF_TYPE(r) (((uint32_t)(r)) >> 28)
#define VK_REF_INDEX(r) (((uint32_t)(r)) & 0x0FFFFFFFu)

/* BVHNode {left, right, bb} (src/accel.rs:52-56).  `left == right` marks the
 * single-object leaf of BVHNode::new (src/accel.rs:102-107): the object is tested
 * twice, which matters for ConstantMedium (two independent free-flight draws). */
typedef struct vk_node {
    float bb_min[3];
    vk_ref left;
    float bb_max[3];
    vk_ref right;
} vk_node; /* 32 B, two 128-bit loads */

typedef struct vk_sphere {
    float center[3];
    float radius; /* may be negative (hollow glass, src/scene.rs:123-127) */
} vk_sphere;      /* 16 B; material in vk_scene_desc.sphere_mat[] */

typedef struct vk_msphere {
    float center0[3];
    float radius;
    float center1[3];
    float time0;
    float time1;
    uint32_t mat;
    uint32_t _pad[2];
} vk_msphere; /* 48 B */

#define VK_RECT_FLIP 0x100u
typedef struct vk_rect {
    float c0, c1, d0, d1; /* bounds on axis0 / axis1 (src/hittable.rs:200-210) */
    float k;              /* plane position on axis2                            */
    uint32_t axes;        /* axis0 | axis1<<2 | axis2<<4 | VK_RECT_FLIP         */
    uint32_t mat;
    uint32_t _pad;
} vk_rect; /* 32 B */

typedef struct vk_box {
    float box_min[3];
    uint32_t mat;
    float box_max[3];
    uint32_t _pad;
} vk_box; /* 32 B; the six sides of Boxy::new (src/hittable.rs:325-353) are implied */

enum {
    VK_X_TRANSLATE = 0, /* a,b,c = offset          src/hittable.rs:500-532 */
    VK_X_ROTATE_X = 1,  /* a = sin, b = cos        src/hittable.rs:631-718 */
    VK_X_ROTATE_Y = 2,  /*                         src/hittable.rs:534-629 */
    VK_X_ROTATE_Z = 3,  /*                         src/hittable.rs:720-807 */
    VK_X_FLIP = 4       /* FlipFace of a non-Rect  src/hittable.rs:294-312 */
};
#define VK_MAX_XFORM_DEPTH 8
typedef struct vk_xform {
    uint32_t kind;
    vk_ref child;
    uint32_t _pad0[2];
    float a, b, c;
    uint32_t _pad1;
} vk_xform; /* 32 B; one record per wrapper level, chains are walked child by child */

typedef struct vk_medium {
    vk_ref boundary;
    float neg_inv_density; /* -1/density, src/hittable.rs:447 */
    uint32_t mat;          /* the Isotropic phase material      */
    uint32_t _pad;
} vk_medium; /* 16 B */

enum {
    VK_M_LAMBERTIAN = 0,    /* src/material.rs:45-109  */
    VK_M_METAL = 1,         /* src/material.rs:111-142 */
    VK_M_DIELECTRIC = 2,    /* src/material.rs:144-207 */
    VK_M_DIFFUSE_LIGHT = 3, /* src/material.rs:209-226 */
    VK_M_ISOTROPIC = 4,     /* src/material.rs:436-465 */
    VK_M_SPECDIFFUSE = 5    /* src/material.rs:467-488 */
};
typedef struct vk_material {
    uint32_t type;
    uint32_t tex;   /* albedo / emit texture index; SPECDIFFUSE: specular material index */
    float param;    /* METAL fuzz | DIELECTRIC ref_idx | SPECDIFFUSE pct                 */
    uint32_t aux;   /* SPECDIFFUSE: diffuse material index                               */
} vk_material;      /* 16 B */

enum {
    VK_TEX_SOLID = 0,   /* src/material.rs:233-242 */
    VK_TEX_CHECKER = 1, /* src/material.rs:244-259 */
    VK_TEX_IMAGE = 2,   /* src/material.rs:261-304 */
    VK_TEX_NOISE = 3    /* src/material.rs:416-434 */
};
typedef struct vk_texture {
    uint32_t type;
    union {
        float rgb[3];                                                  /* SOLID   */
        struct { uint32_t odd, even, _p; } checker;                    /* CHECKER */
        struct { uint32_t texel_offset, width, height; } image;        /* IMAGE: RGB8, BPP=3 */
        struct { uint32_t perlin; float scale; uint32_t _p; } noise;   /* NOISE   */
    };
} vk_texture; /* 16 B */

/* Perlin tables (src/material.rs:306-311), generated on the host (:357-377). */
typedef struct vk_perlin {
    float ranvec[256][3];
    uint8_t perm_x[256];
    uint8_t perm_y[256];
    uint8_t perm_z[256];
} vk_perlin;

typedef struct vk_scene_desc {
    uint32_t api_version; /* VK_API_VERSION */
    vk_ref root;          /* the world: `BVHNode::new(&mut config.world)` src/main.rs:168 */

    const vk_node* nodes;        uint32_t n_nodes;
    const vk_sphere* spheres;    const uint32_t* sphere_mat; uint32_t n_spheres;
    const vk_msphere* mspheres;  uint32_t n_mspheres;
    const vk_rect* rects;        uint32_t n_rects;
    const vk_box* boxes;         uint32_t n_boxes;
    const vk_xform* xforms;      uint32_t n_xforms;
    const vk_medium* media;      uint32_t n_media;

    const vk_ref* lights;        uint32_t n_lights; /* SceneConfig.lights src/scene.rs:19 */

    const vk_material* materials; uint32_t n_materials;
    const vk_texture* textures;   uint32_t n_textures;
    const uint8_t* texels;        uint64_t n_texel_bytes;
    const vk_perlin* perlins;     uint32_t n_perlins;
} vk_scene_desc;

/* Camera (src/main.rs:56-68): the ten fields, in declaration order. */
typedef struct vk_camera {
    float origin[3];
    float lower_left_corner[3];
    float horizontal[3];
    float vertical[3];
    float u[3], v[3], w[3];
    float lens_radius;
    float time0, time1;
} vk_camera; /* 24 floats */

/* AUTO picks by the evidence recorded in DESIGN.md / profiles/.  MEGAKERNEL = one lane, one path
 * (persistent threads, path regeneration); WAVEFRONT = generate / extend / shade as separate kernels
 * over a slot pool in device memory; STAGED = the persistent megakernel with the wavefront's stages
 * and material sort inside each CTA (slot pool in shared memory); WARPQ = the same stages inside each
 * WARP: per-warp slot pool and per-class queues in shared memory, no barrier anywhere; STEPQ = warp
 * queues for BVH scenes with the traversal itself cut into queued steps (node visit / sphere / box /
 * other leaves), traversal state in shared memory (a flat-program scene runs WARPQ). */
enum { VK_VARIANT_AUTO = 0, VK_VARIANT_MEGAKERNEL = 1, VK_VARIANT_WAVEFRONT = 2, VK_VARIANT_STAGED = 3, VK_VARIANT_WARPQ = 4,
       VK_VARIANT_STEPQ = 5 };
enum {
    VK_FLAG_STRICT_MATH = 1u, /* no FMA contraction, IEEE div/sqrt, division slab test:
                                 the op sequence of the reference, for hit parity    */
    VK_FLAG_FORCE_BVH = 2u,   /* traverse the BVH even when the scene is small enough for
                                 the flat (divergence-free) traversal program         */
    VK_FLAG_LEGACY_SCATTER = 4u, /* the book-1/2 integrator of the reference's legacy `Material::scatter`
                                 methods (src/material.rs:21-28, 85-90, 118-132, 150-175, 215-217,
                                 442-446): no light list, no PDFs, `emitted + attenuation *
                                 ray_color(scattered)`.  HEAD itself cannot render a scene without
                                 lights (`choose().unwrap()` panics, src/hittable.rs:431)          */
    VK_FLAG_SKY_BACKGROUND = 8u  /* a missed ray returns the book-1 sky (1-t)*white + t*(0.5,0.7,1),
                                 t = 0.5*(unit(d).y + 1) (sample/inoneweekend.png) instead of
                                 `background` (src/main.rs:124)                                    */
};

/* The constants of src/main.rs:28-29,171-172 and the choices the reference leaves
 * to its (unseeded) RNG, as parameters. */
typedef struct vk_render_params {
    uint32_t width, height;
    uint32_t spp;       /* SAMPLES_PER_PIXEL: the divisor of the mean (main.rs:196)     */
    uint32_t spp_begin; /* this call renders global samples [spp_begin, spp_begin+spp_count) */
    uint32_t spp_count; /* 0 == all of them (spp - spp_begin)                            */
    uint32_t max_depth; /* MAX_DEPTH, `depth > MAX_DEPTH` semantics (main.rs:126): a path
                         * traces at most max_depth segments.  Must be >= 1: ray_color starts
                         * at depth 1, so 0 is a black frame with no rays, and every render
                         * call refuses it with VK_ERR_INVALID.                          */
    uint64_t seed;      /* Philox4x32-10 key                                             */
    float background[3];/* src/main.rs:124 (always 0 at HEAD)                            */
    uint32_t variant;   /* VK_VARIANT_*                                                  */
    uint32_t flags;     /* VK_FLAG_*                                                     */
} vk_render_params;

typedef struct vk_stats {
    uint64_t paths;           /* samples started = W*H*spp_count                         */
    uint64_t rays;            /* world.hit() segment queries from ray_color (main.rs:130)*/
    uint64_t dropped_samples; /* non-finite samples filtered (main.rs:191-194)           */
    float ms_kernels;         /* CUDA-event time of the render kernels                   */
    float ms_total;           /* CUDA-event time incl. D2H of the image (vk_render)      */
    uint32_t variant;         /* variant that ran                                        */
    uint32_t launches;        /* kernels launched by this call                           */
    uint64_t node_visits;     /* BVH nodes fetched (wide nodes: one fetch tests two boxes) */
    uint64_t prim_tests;      /* primitive / instance / medium tests                      */
} vk_stats;

typedef struct vk_ray {
    float origin[3];
    float direction[3];
    float time;
    float tmin, tmax;
} vk_ray; /* 36 B */

/* HitRec (src/hittable.rs:11-20) plus the primitive id the reference lacks. */
typedef struct vk_hit {
    vk_ref prim;    /* leaf record that produced the hit; VK_REF_NONE == miss */
    uint32_t face;  /* BOX: side index 0..5 in Boxy::new order; else 0        */
    uint32_t mat;
    uint32_t front;
    float t;
    float p[3];
    float normal[3];
    float u, v;
    uint32_t _pad;
} vk_hit; /* 56 B */

#define VK_MEDIUM_XI_SLOTS 8 /* vk_intersect's injected table: slot = medium index * 2 + second-visit; scenes of up to 4 media */

typedef struct vk_ctx vk_ctx;

/* Create a context on CUDA device `device`.  Replaces nothing in the reference
 * (it has no device); owns the stream, device scene and accumulation buffers. */
int vk_create(int device, vk_ctx** out);
void vk_destroy(vk_ctx* ctx);
/* Message of the last failure on `ctx` (or of the last failed vk_create if NULL). */
const char* vk_last_error(const vk_ctx* ctx);

/* Copy a flattened scene to the device (host arrays are borrowed for the call).
 * Replaces the `Arc<BVHNode>` world / `Arc<Vec<..>>` lights handed to the loop at
 * src/main.rs:168-169. */
int vk_scene_upload(vk_ctx* ctx, const vk_scene_desc* scene);

/* Host-only: validate a flattened scene and plan its device layout exactly as vk_scene_upload would,
 * without a device.  Reports what the upload would build (and lets CPU tests cover the validator, the
 * 4-wide BVH collapse and the flat-program builder).  Same return codes as vk_scene_upload; the message
 * goes to err (nullable). */
typedef struct vk_scene_info {
    uint32_t flat_entries;         /* primitives in the flat traversal program, 0 = the BVH is traversed   */
    uint32_t flat_segments;        /* world frame + instance frames                                        */
    uint32_t flat_subtrees;        /* hybrid program: homogeneous subtrees kept as BVH entries (0 = pure)  */
    uint32_t simple;               /* 1 = the trimmed ("simple scene") build of the staged kernel applies  */
    uint32_t wide_nodes;           /* 4-wide nodes made from the reference's binary nodes                  */
    uint32_t wide_levels_world;    /* 4-wide levels of the world BVH / of the deepest instanced sub-BVH     */
    uint32_t wide_levels_instance;
    uint32_t stack_need;           /* traversal stack entries needed (<= 96)                               */
    uint32_t dynamic_megakernel;   /* 1 = BVH large enough for the dynamic re-fill megakernel               */
    uint32_t flat_boxes;           /* Boxy entries of the flat program (render build: one slab test each)   */
    uint32_t flat_direct;          /* hit-table entries whose HitRec the shade stage writes down directly   */
    uint32_t flat_shape;           /* 0, or the flat program's shape the warp-queue kernel is compiled for  */
} vk_scene_info;
int vk_scene_check(const vk_scene_desc* scene, vk_scene_info* info, char* err, size_t err_len);

/* The sample loop, src/main.rs:181-198.  out_rgb: W*H*3 floats, pixel i = y*W+x,
 * row 0 = bottom (main.rs:182-183), linear mean over `spp` (main.rs:196).
 * out_sumsq (nullable): per channel sum of squares of the kept samples.  Host buffers. */
int vk_render(vk_ctx* ctx, const vk_camera* cam, const vk_render_params* params,
              float* out_rgb, float* out_sumsq, vk_stats* stats);

/* The sample loop followed by the output conversion of src/main.rs:201-214 on the device: every
 * channel goes through Vec3::to_color (src/vec3.rs:54-61: (256 * clamp(sqrt(c), 0, 0.999)) as u32, NaN
 * -> 0) and the rows are written top-down (y = height-1 first, main.rs:209), i.e. out_rgb8 holds the
 * W*H*3 numbers of the reference's P3 file in file order.  Only a quarter of the bytes cross PCIe.
 * A turntable (RotatingCamera, src/scene.rs:65-91) calls this once per camera with the scene resident. */
int vk_render_rgb8(vk_ctx* ctx, const vk_camera* cam, const vk_render_params* params,
                   uint8_t* out_rgb8, vk_stats* stats);

/* K cameras of one scene in one launch.  Frame f uses cams[f] and Philox key params->seed + f (the rule of
 * vecchio_gpu_render --seed); every other field of params applies to every frame.  Frame f of the output, at offset
 * f * W*H*3, is what vk_render / vk_render_rgb8 return for (cams[f], seed + f) ON THE SAME KERNEL, bit for bit.
 * The frames' units share the warps (frame-major: the batch drains once), and VK_VARIANT_AUTO decides on the batch's
 * path count n_frames * W * H * spp_count, so a batch may run another kernel than its frames would one by one (config 1's
 * turntable, 400x225x16: the step queues from 3 frames on, the lane megakernel for one).  With VK_FLAG_STRICT_MATH every
 * kernel computes the reference's operation sequence and the batch equals the single-frame calls bit for bit whatever
 * ran; in the render build each kernel contracts FMAs its own way, so there the guarantee needs an explicit variant:
 * with AUTO a batch that changes kernel renders the same estimate with other rounding (individual samples can differ).
 * stats: totals of the batch (paths, rays, dropped samples, kernel time) and
 * the variant that ran.  No sums of squares (vk_render keeps them).  n_frames == 1 is vk_render / vk_render_rgb8.
 * Errors, before anything is launched: VK_ERR_INVALID for n_frames == 0, a null pointer, a camera with
 * time0 >= time1 (the message names the frame) or n_frames * W*H*3 >= 2^31; VK_ERR_OOM when the batch's accumulators
 * cannot be allocated; VK_ERR_UNSUPPORTED for VK_VARIANT_STAGED / VK_VARIANT_WAVEFRONT with n_frames > 1;
 * VK_ERR_NO_SCENE without a scene. */
int vk_render_frames(vk_ctx* ctx, const vk_camera* cams, uint32_t n_frames, const vk_render_params* params,
                     float* out_rgb, vk_stats* stats);
int vk_render_frames_rgb8(vk_ctx* ctx, const vk_camera* cams, uint32_t n_frames, const vk_render_params* params,
                          uint8_t* out_rgb8, vk_stats* stats);

/* Adaptive sampling: every pixel renders until its displayed noise is below max_error, or until params->spp samples.
 * Passes: pass 0 renders global samples [0, pass_spp) of every pixel; pass k renders [k*pass_spp, min((k+1)*pass_spp, spp))
 * of every pixel still active.  A pixel therefore ends with n_p in {pass_spp, 2*pass_spp, ..} or n_p = spp samples, and
 * they are exactly its samples [0, n_p): its mean is, bit for bit, what vk_render returns for that pixel with spp = n_p on
 * the same kernel (Philox is keyed by pixel and global sample, the accumulators are integers).
 * Stopping rule, after each pass, per channel of the pixel (in the reference's output units, Vec3::to_color's sqrt x 256):
 *     m = sum / n,  se = sqrt(max(Q / n - m^2, 0) / (n - 1))   (Q: sum of squares),
 *     e = 128 * (sqrt(max(m + se, 0)) - sqrt(max(m - se, 0))),  half the width of sqrt(m +- se) in 8-bit steps;
 * the pixel stops when the largest e of its three channels is <= max_error, or when n == spp.  max_error == 0 never stops
 * early; a pixel with one sample (pass_spp == 1, pass 0) has no standard error and renders on.
 * The squares behind the rule are 64-bit fixed-point sums (2^32 units per 1.0, the sample's channel clamped to 255 first:
 * the clamp touches the statistic only, never the image), exact and order independent; this bounds spp to 65536.
 * The decision is a stated function of the integer state (sum S: int64 at 2^30 units per 1.0, Q: uint64, n), every step
 * an IEEE double operation rounded to nearest:
 *     m = (double)S * 2^-30 / n,  q = (double)Q * 2^-32 / n   (the conversions round to nearest),
 *     v = fma(-m, m, q)   (q - m^2 with ONE rounding),
 *     se = sqrt(max(v, 0) / (n - 1)),  e_c = (sqrt(max(m + se, 0)) - sqrt(max(m - se, 0))) * 128,
 *     e = max(0, e_R, e_G, e_B), and the test is e <= (double)max_error;
 * out_error maps hold (float)e.  tests/adaptive_model.py restates it on the host, bit for bit.
 * The rule looks at the samples, so the estimate is slightly BIASED: pixels that happen to look smooth stop early.
 * Kernel: VK_VARIANT_AUTO decides once, by vk_render's rule on pass 0's path count W*H*pass_spp, and every pass runs that
 * kernel, so a pass boundary never changes rounding (render build included).
 * out_rgb: the means sum / n_p in vk_render's layout; out_rgb8: to_color of the same means, top-down like vk_render_rgb8;
 * out_spp (nullable): n_p, W*H in the order of the image it accompanies.  stats: paths = sum of n_p; rays, dropped
 * samples, ms_kernels and launches are totals over all passes; variant is the kernel that ran.  Each pass costs one 4-byte
 * D2H of the active count and a stream synchronisation.  One frame on one device (a batch of frames:
 * vk_render_frames_adaptive; several devices: vk_multi_render_adaptive_rgb8).
 * Errors, before anything is launched: VK_ERR_INVALID for pass_spp == 0, max_error negative or NaN, spp_begin != 0,
 * spp_count not 0 or spp, spp > 65536, and every check of vk_render; VK_ERR_UNSUPPORTED for VK_VARIANT_STAGED /
 * VK_VARIANT_WAVEFRONT; VK_ERR_NO_SCENE without a scene. */
int vk_render_adaptive(vk_ctx* ctx, const vk_camera* cam, const vk_render_params* params,
                       uint32_t pass_spp, float max_error,
                       float* out_rgb, uint32_t* out_spp, vk_stats* stats);
int vk_render_adaptive_rgb8(vk_ctx* ctx, const vk_camera* cam, const vk_render_params* params,
                            uint32_t pass_spp, float max_error,
                            uint8_t* out_rgb8, uint32_t* out_spp, vk_stats* stats);

/* Adaptive sampling of K cameras of one scene: vk_render_adaptive's passes and stopping rule over a batch, as
 * vk_render_frames batches vk_render.  Frame f uses cams[f] and Philox key params->seed + f.  Pass k renders global samples
 * [k*pass_spp, min((k+1)*pass_spp, spp)) of every pixel still active in ANY frame, in ONE launch over one list of the active
 * pixels of all frames (the frames share the warps and one drain tail per pass); the rule is applied per pixel, unchanged,
 * and a frame whose pixels have all stopped simply has no entries left.  The call ends when no pixel is active or spp is
 * reached; each pass costs one 4-byte D2H and a stream synchronisation.
 * Frame f's image AND counts equal, bit for bit, what vk_render_adaptive(_rgb8) returns for (cams[f], seed + f, pass_spp,
 * max_error) ON THE SAME KERNEL (a pixel's decision depends on its own integer sums only).  The same-kernel caveat is
 * vk_render_frames': VK_VARIANT_AUTO decides once, on the batch's pass-0 path count n_frames * W*H * min(pass_spp, spp), so a
 * batch may run another kernel than its frames would one by one.  With VK_FLAG_STRICT_MATH the frames are equal whatever
 * ran.  In the render build each compiled kernel contracts multiply-adds its own way and a batch runs kernels of its own, so
 * there equality needs the same variant and is not bit for bit everywhere: the lane megakernel for flat scenes lit by one
 * rect (Cornell box) gives the same counts but rounds some pixels differently.
 * Like vk_render_adaptive's, the estimate is slightly BIASED: pixels that happen to look smooth stop early.
 * out_rgb: n_frames planes of W*H*3 means, frame f at offset f * W*H*3, rows bottom-up (vk_render_frames' layout);
 * out_rgb8: each frame top-down (vk_render_frames_rgb8's layout); out_spp (nullable): n_frames * W*H counts in the row order
 * of the image they accompany.  stats: paths = sum of n_p over all frames; rays, dropped samples, ms_kernels and launches
 * are totals over all passes; variant is the kernel that ran.  n_frames == 1 is vk_render_adaptive(_rgb8).
 * Errors, before anything is launched: every error of vk_render_frames (n_frames == 0, a null pointer, a bad camera with
 * the frame named, n_frames * W*H*3 >= 2^31, VK_ERR_OOM) and of vk_render_adaptive (pass_spp, max_error,
 * spp_begin / spp_count, spp > 65536); VK_ERR_UNSUPPORTED for VK_VARIANT_STAGED / VK_VARIANT_WAVEFRONT; VK_ERR_NO_SCENE
 * without a scene. */
int vk_render_frames_adaptive(vk_ctx* ctx, const vk_camera* cams, uint32_t n_frames, const vk_render_params* params,
                              uint32_t pass_spp, float max_error,
                              float* out_rgb, uint32_t* out_spp, vk_stats* stats);
int vk_render_frames_adaptive_rgb8(vk_ctx* ctx, const vk_camera* cams, uint32_t n_frames, const vk_render_params* params,
                                   uint32_t pass_spp, float max_error,
                                   uint8_t* out_rgb8, uint32_t* out_spp, vk_stats* stats);

/* Adaptive render sessions: vk_render_frames_adaptive's passes and stopping rule, with the state kept between calls so a
 * render can be tightened step by step (a preview at max_error 8 that becomes the final frame at 1 without repeating a
 * sample), saved and resumed.  A session renders K >= 1 cameras of the context's scene: frame f uses cams[f] and Philox key
 * params->seed + f, and every pass renders pass_spp = M samples (the last one up to the cap).  It is moved by targets: */
typedef struct vk_adaptive_target {
    uint32_t spp;     /* cap: no pixel renders more than spp samples                                */
    uint32_t min_spp; /* floor: a pixel does not stop before n >= min_spp (the cap still wins)      */
    float max_error;  /* the stopping rule's bound in 8-bit steps; 0 = never stop early            */
} vk_adaptive_target;
typedef struct vk_adaptive_session vk_adaptive_session;

/* The rule, checked at pass boundaries only: a pixel at n samples stops when n == spp, or when n >= min_spp, n > 1 and the
 * largest channel error e <= max_error (e as vk_render_adaptive states it).  With min_spp = 0 it is the one-shot calls'
 * rule.  A pixel's count is therefore on the pass grid (a multiple of M) or equal to a cap.
 * Tightening: a target T2 may follow the target T1 the session last reached only if
 *     T2.max_error <= T1.max_error, where 0 is the tightest value (after 0 only 0 may follow);
 *     T2.min_spp >= T1.min_spp;
 *     T2.spp >= T1.spp, and T2.spp > T1.spp only when T1.spp is a multiple of M (pixels stopped at the old cap go on along
 *     the pass grid);
 *     T2.spp <= params->spp, the session's limit.
 * A fresh session has reached no target and accepts any first target within its limit.
 * Guarantee: after any sequence of tightening targets ending in T, the state (sums, squares, counts) is bit for bit the
 * state of a fresh session refined once to T.  (A pixel that stopped at n1 under T1 went on at every earlier grid point b:
 * b < T1.min_spp <= T2.min_spp or e(b) > T1.max_error >= T2.max_error, so a fresh T2 render also reaches n1 with the same
 * integer sums; from n1 on both apply T2's rule to the same integers.)  A fresh session refined to {params->spp, 0, E}
 * equals vk_render_adaptive(_rgb8) (K = 1) or vk_render_frames_adaptive(_rgb8) (K > 1) at max_error = E in image, counts and
 * stats.paths, in both math builds: it runs the same kernels.
 * Sessions borrow their context: destroy them before the context.  Other calls on the context (vk_render, the one-shot
 * adaptive calls, other sessions) may run between a session's calls and do not touch its state.  Several GPUs:
 * vk_adaptive_begin_shard on each, or vk_multi_adaptive_begin over a vk_multi.
 * Errors are reported through vk_last_error of the context. */

/* Begins a session: every check of vk_render_frames_adaptive (params->spp is the session's limit, <= 65536; spp_begin
 * must be 0 and spp_count 0 or spp; pass_spp >= 1; VK_ERR_UNSUPPORTED for VK_VARIANT_STAGED / VK_VARIANT_WAVEFRONT;
 * VK_ERR_NO_SCENE without a scene), then the session's own device buffers (sums, squares, counts and pass lists for
 * n_frames * W*H pixels, zeroed) and its kernel: VK_VARIANT_AUTO decides here, once, by the one-shot rule on
 * n_frames * W*H * min(pass_spp, spp) paths.  The cameras and params are copied. */
int vk_adaptive_begin(vk_ctx* ctx, const vk_camera* cams, uint32_t n_frames, const vk_render_params* params,
                      uint32_t pass_spp, vk_adaptive_session** out);

/* Shard sessions: a session that renders only the pixels shard `shard` of n_shards owns, so that n_shards devices (or
 * processes) can split one adaptive render between them without any traffic until the image is read.
 * Ownership: with g the batch-wide pixel index f*W*H + y*W + x, pixel g belongs to shard (g / VK_SHARD_RUN) mod n_shards.
 * A run of VK_SHARD_RUN = 32 pixels is one warp's list entries and one lane-megakernel item, so a shard's lists keep the
 * alignment and the camera-ray coherence of the unsharded lists, and the fine interleaving spreads noisy regions evenly.
 * The session is an ordinary vk_adaptive_session: refine, read, read_rgb8, export, import, variant and destroy take it.
 * Its buffers are full size (n_frames * W*H) and indices stay batch-wide.  Pixels it does not own are never rendered:
 * their sums, squares and counts stay 0 and read like any pixel without samples (count 0, mean 0/0 = NaN, rgb8 0, error
 * +inf).  Its kernel is the unsharded session's: VK_VARIANT_AUTO decides on the whole batch's
 * n_frames * W*H * min(pass_spp, spp) paths, not on the shard's share.
 * A shard that owns no pixel (n_frames * W*H <= 32 * shard) is legal: its refines render nothing, add 0 paths and still
 * reach their target.  vk_adaptive_import also refuses (VK_ERR_INVALID, the state untouched) any non-zero sum, square or
 * count on a pixel the shard does not own.
 * Guarantee: a pixel's decisions depend on its own integer state only and Philox is keyed by (pixel, global sample), so an
 * owned pixel ends every refine with the integers it has in the unsharded session.  For any sequence of tightening targets,
 * the sum over shards k = 0 .. n_shards-1 of their exports equals the unsharded session's export bit for bit (and paths add
 * up likewise).  Shard 0 of 1 is vk_adaptive_begin.
 * Errors: those of vk_adaptive_begin, and VK_ERR_INVALID for n_shards == 0 or shard >= n_shards. */
#define VK_SHARD_RUN 32
int vk_adaptive_begin_shard(vk_ctx* ctx, const vk_camera* cams, uint32_t n_frames, const vk_render_params* params,
                            uint32_t pass_spp, uint32_t shard, uint32_t n_shards, vk_adaptive_session** out);

/* Renders until `target` is reached.  A pixel below the new cap that the new rule lets go on renders on from its count;
 * the passes run level by level (a level is a count on the pass grid: 0, M, 2M, ..), each pass one launch over the pixels
 * at that level, and a level without pixels costs nothing.  One small read-back per refine, plus one per pass as in the
 * one-shot calls.  stats (nullable) are for this refine only: paths = samples added; rays, dropped samples, ms_kernels and
 * launches as the one-shot calls count them.
 * VK_ERR_INVALID, the state untouched: a null target; target.spp 0 or above the limit; max_error negative or NaN; a target
 * that does not tighten the one reached (see above); the scene changed (re-uploaded) since the session began; an earlier
 * refine or import that failed part way (the state is lost: read, export and refine refuse until a successful
 * vk_adaptive_import replaces the whole state, e.g. from a checkpoint; otherwise only destroy is left). */
int vk_adaptive_refine(vk_adaptive_session* session, const vk_adaptive_target* target, vk_stats* stats);

/* The state's image, in the one-shot calls' layouts: vk_adaptive_read gives the means sum / n in vk_render_frames' layout
 * (rows bottom-up), vk_adaptive_read_rgb8 to_color of them, each frame top-down.  out_spp (nullable): the counts and
 * out_error (nullable): per pixel the largest channel e as the rule sees it, as float, +inf where n < 2; both
 * n_frames * W*H in the row order of the image they accompany.  Reading does not change the state. */
int vk_adaptive_read(vk_adaptive_session* session, float* out_rgb, uint32_t* out_spp, float* out_error);
int vk_adaptive_read_rgb8(vk_adaptive_session* session, uint8_t* out_rgb8, uint32_t* out_spp, float* out_error);

/* The raw state, for checkpoints: sums (signed fixed point, 2^30 units per 1.0) and squares (unsigned fixed point, 2^32
 * units per 1.0, each sample's channel clamped to 255 first), n_frames * W*H * 3 each, and counts,
 * n_frames * W*H, all in the accumulators' order (frame by frame, rows bottom-up); reached (nullable) is the last target
 * reached, all zero for a session that has reached none. */
int vk_adaptive_export(vk_adaptive_session* session, int64_t* sums, uint64_t* squares, uint32_t* counts,
                       vk_adaptive_target* reached);
/* Replaces the state by exported arrays of a session with the same scene, cameras, params, pass_spp and kernel (the library
 * cannot see those: the caller keeps them with the checkpoint).  VK_ERR_INVALID, the state untouched, unless reached.spp is
 * within the limit, reached.max_error >= 0, and every count is <= reached.spp and on the grid (a multiple of pass_spp or
 * reached.spp; a count of 0 with zero sums and squares).  reached.spp == 0 is a state that reached no target.  Because
 * it replaces the whole state, a successful import is also how a session recovers after a refine or import that failed
 * part way. */
int vk_adaptive_import(vk_adaptive_session* session, const int64_t* sums, const uint64_t* squares, const uint32_t* counts,
                       const vk_adaptive_target* reached);

/* The kernel (VK_VARIANT_*) every pass of the session runs, fixed by vk_adaptive_begin: part of a checkpoint's identity,
 * since the render build's kernels may round differently.  0 for a null session. */
uint32_t vk_adaptive_variant(const vk_adaptive_session* session);

/* Frees the session's buffers.  Before vk_destroy of its context. */
void vk_adaptive_destroy(vk_adaptive_session* session);

/* Same loop, device-resident result: writes per-pixel SUMS (not means) of samples
 * [spp_begin, spp_begin+spp_count) to d_sum (and d_sumsq, nullable), both device
 * pointers of W*H*3 floats, enqueued on the context stream; synchronised before return
 * only when stats != NULL.  This is the per-GPU spp slice; slices are combined by one NCCL
 * reduce. */
int vk_render_device(vk_ctx* ctx, const vk_camera* cam, const vk_render_params* params,
                     float* d_sum, float* d_sumsq, vk_stats* stats);

/* d_rgb[i] = d_sum[i] / spp on the device (main.rs:196), after the reduce.  Asynchronous on the
 * context stream. */
int vk_finalize_device(vk_ctx* ctx, const float* d_sum, float* d_rgb, size_t n_floats,
                       uint32_t spp);

/* Enqueue all following work on `stream` (a cudaStream_t of the caller, e.g. the one its NCCL
 * reduce runs on); NULL restores the context's own stream. */
int vk_set_stream(vk_ctx* ctx, void* stream);

/* Counters accumulated since the last read (paths, rays, dropped samples, kernel launches);
 * synchronises the stream.  vk_render_device with stats == NULL is fully asynchronous and leaves
 * its counts to be collected here. */
int vk_flush_stats(vk_ctx* ctx, vk_stats* stats);

/* One context over several GPUs of a node: what replaces the rayon pool of src/main.rs:181 when the host has more
 * than one device.  The frame's samples are split by GLOBAL sample index (device k of N renders
 * [k * count / N, (k + 1) * count / N) of the requested range, for every pixel), every device keeps its slice in
 * 64-bit fixed-point accumulators, and device devices[0] adds its peers' accumulators to its own with a kernel that
 * reads them over NVLink (peer-mapped memory; no communicator, no host staging).  Integer addition: the frame is
 * bit-identical to the frame one GPU renders for the same seed, whatever N.  Same conventions as the single-device
 * calls; vk_multi_last_error(NULL) reports a failed vk_multi_create. */
typedef struct vk_multi vk_multi;
int vk_multi_create(const int* devices, int n_devices, vk_multi** out);
void vk_multi_destroy(vk_multi* m);
const char* vk_multi_last_error(const vk_multi* m);
int vk_multi_device_count(const vk_multi* m);
int vk_multi_scene_upload(vk_multi* m, const vk_scene_desc* scene);            /* the scene is replicated on every device */
int vk_multi_render(vk_multi* m, const vk_camera* cam, const vk_render_params* params, float* out_rgb, float* out_sumsq,
                    vk_stats* stats);                                           /* vk_render over all devices              */
int vk_multi_render_rgb8(vk_multi* m, const vk_camera* cam, const vk_render_params* params, uint8_t* out_rgb8,
                         vk_stats* stats);                                      /* vk_render_rgb8 over all devices         */
int vk_multi_render_frames_rgb8(vk_multi* m, const vk_camera* cams, uint32_t n_frames, const vk_render_params* params,
                                uint8_t* out_rgb8, vk_stats* stats);            /* vk_render_frames_rgb8 over all devices  */

/* Adaptive sessions over all devices of a vk_multi: the vk_adaptive_* calls with the same meaning and arguments.  Adaptive
 * sampling splits PIXELS, not samples (a pixel's decision after each pass needs the sums of all its samples): device k
 * runs shard k of N (vk_adaptive_begin_shard), the existing pass loop over the pixels it owns.  A refine runs the devices'
 * pass loops at once, one host thread per device inside the call, all joined before it returns.  stats: paths, rays,
 * dropped samples and launches summed over the devices, ms_kernels the slowest device's, variant the shared kernel.
 * A read or an export after a refine or an import first gathers every pixel's sums, squares and count from the device
 * that owns it into one state on devices[0] (one kernel reading the peers' memory over NVLink, 52 bytes a pixel), then
 * reads it as vk_adaptive_read* / vk_adaptive_export do.  An import checks the whole state as vk_adaptive_import does and
 * gives each device the pixels it owns; a refused import changes nothing.  After a refine or import that failed part way
 * on any device the session refuses everything but import and destroy.  Errors: vk_multi_last_error of the vk_multi.
 * Guarantee: the image, counts, error map, export and stats.paths equal those of a one-GPU session with the same
 * arguments, bit for bit, in both math builds: every device runs the one-GPU session's kernel on the same integers.  So an
 * export of either resumes in the other.  Destroy the session before the vk_multi.
 * The balance is static: the slowest shard sets the time of every refine. */
typedef struct vk_multi_adaptive_session vk_multi_adaptive_session;
int vk_multi_adaptive_begin(vk_multi* m, const vk_camera* cams, uint32_t n_frames, const vk_render_params* params,
                            uint32_t pass_spp, vk_multi_adaptive_session** out);
int vk_multi_adaptive_refine(vk_multi_adaptive_session* session, const vk_adaptive_target* target, vk_stats* stats);
int vk_multi_adaptive_read(vk_multi_adaptive_session* session, float* out_rgb, uint32_t* out_spp, float* out_error);
int vk_multi_adaptive_read_rgb8(vk_multi_adaptive_session* session, uint8_t* out_rgb8, uint32_t* out_spp, float* out_error);
int vk_multi_adaptive_export(vk_multi_adaptive_session* session, int64_t* sums, uint64_t* squares, uint32_t* counts,
                             vk_adaptive_target* reached);
int vk_multi_adaptive_import(vk_multi_adaptive_session* session, const int64_t* sums, const uint64_t* squares,
                             const uint32_t* counts, const vk_adaptive_target* reached);
uint32_t vk_multi_adaptive_variant(const vk_multi_adaptive_session* session);
void vk_multi_adaptive_destroy(vk_multi_adaptive_session* session);
/* vk_render_adaptive_rgb8 / vk_render_frames_adaptive_rgb8 over all devices: begin, one refine to {spp, 0, max_error} and
 * read_rgb8 on a session the vk_multi keeps; the same bytes, counts and stats.paths as on one GPU.  (Float means, error
 * maps and exports: through a session.)  stats.ms_total: the call's wall time. */
int vk_multi_render_adaptive_rgb8(vk_multi* m, const vk_camera* cam, const vk_render_params* params, uint32_t pass_spp,
                                  float max_error, uint8_t* out_rgb8, uint32_t* out_spp, vk_stats* stats);
int vk_multi_render_frames_adaptive_rgb8(vk_multi* m, const vk_camera* cams, uint32_t n_frames, const vk_render_params* params,
                                         uint32_t pass_spp, float max_error, uint8_t* out_rgb8, uint32_t* out_spp,
                                         vk_stats* stats);

/* Parity hook: closest hit of `world.hit(&r, tmin, tmax)` (src/accel.rs:58-83) for
 * a batch of rays.  medium_xi (nullable): n * VK_MEDIUM_XI_SLOTS uniform variates
 * for ConstantMedium::hit's free-flight draw (src/hittable.rs:473). */
int vk_intersect(vk_ctx* ctx, const vk_ray* rays, size_t n, const float* medium_xi,
                 uint32_t flags, vk_hit* out);

/* Parity hook for the SHADING half of the path, next to vk_intersect for the geometry half: one call of the
 * device functions behind `Material::scatter_with_pdf` / `scattering_pdf` / `emitted` (src/material.rs:92-108,
 * 134-141, 177-206, 218-225, 448-487), `Texture::value` (:238-303, 430-433), the light list's `pdf_value` /
 * `random` (src/hittable.rs:104-134, 271-291, 371-377, 420-433) and the mixture estimator that ties them
 * together in `ray_color` (src/main.rs:131-149) -- on the uploaded scene's materials, textures and lights, with
 * the variates SUPPLIED so that the oracle can be fed the same ones.
 *   VK_EVAL_BOUNCE         one pass of ray_color's body after world.hit() returned the given HitRec:
 *                          beta starts at (1,1,1), L at 0; out = continue?, scattered ray, weight, emission
 *   VK_EVAL_BOUNCE_LEGACY  the same for the legacy `Material::scatter` integrator
 *   VK_EVAL_TEXTURE        textures[index].value(u, v, p) -> beta
 *   VK_EVAL_LIGHTS_PDF     lights.pdf_value(p, dir) -> value            (`impl Hittable for Vec<..>`, :420-427)
 *   VK_EVAL_LIGHT_RANDOM   lights[index].random(p) with xi[0..2] -> out_d */
enum { VK_EVAL_BOUNCE = 0, VK_EVAL_BOUNCE_LEGACY = 1, VK_EVAL_TEXTURE = 2, VK_EVAL_LIGHTS_PDF = 3, VK_EVAL_LIGHT_RANDOM = 4 };
typedef struct vk_eval {
    uint32_t op;
    uint32_t index;                     /* BOUNCE*: material | TEXTURE: texture | LIGHT_RANDOM: entry of the light list */
    float ray_o[3], ray_d[3], ray_time; /* BOUNCE*: the ray that was traced                                              */
    float p[3], normal[3], t, u, v;     /* BOUNCE*: the HitRec | TEXTURE: u, v, p | LIGHT*: p = the origin               */
    uint32_t front;
    float dir[3];                       /* LIGHTS_PDF: the direction                                                    */
    uint32_t xi[5];                     /* BOUNCE*: xi[0..3] the bounce's four 32-bit variates (gen::<f32>() takes the
                                           top 24 bits, gen_range the top 23), xi[4] SpecDiffuse's choice;
                                           LIGHT_RANDOM: xi[0..2]                                                       */
    /* results */
    uint32_t alive;                     /* BOUNCE*: the path continues with (out_o, out_d, out_time)                     */
    uint32_t valid;                     /* BOUNCE*: 0 = the reference's sample is non-finite here (dropped, main.rs:192) */
    float out_o[3], out_d[3], out_time;
    float beta[3];                      /* BOUNCE*: path weight after the bounce | TEXTURE: the colour                   */
    float L[3];                         /* BOUNCE*: radiance added by this hit                                           */
    float value;                        /* LIGHTS_PDF                                                                   */
} vk_eval; /* 43 words */
int vk_eval_batch(vk_ctx* ctx, vk_eval* recs, size_t n, uint32_t flags /* VK_FLAG_STRICT_MATH */);

/* Microbenchmarks for the roofline denominators the driver does not measure:
 * dependent-free FFMA throughput (TFLOP/s) and L2-resident read bandwidth (GB/s). */
int vk_measure_peaks(vk_ctx* ctx, float* fp32_tflops, float* l2_gbs);

/* Device properties for reporting. */
int vk_device_info(vk_ctx* ctx, int* sm_count, int* clock_khz, char* name, size_t name_len);

#ifdef __cplusplus
}
#endif
#endif /* VECCHIO_GPU_H */
