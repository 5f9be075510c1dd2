// vk_internal.h -- device-side scene layout and the launcher interface between vk_api.cu (context,
// upload, C ABI) and vk_kernels.cu (device code, compiled twice: namespace vkfast with FMA
// contraction, namespace vkstrict with -fmad=false and the reference's op sequence).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/vecchio_gpu.h"

// Device references add two things to vk_ref: bit 27 marks the SECOND visit of a single-object BVH
// leaf that holds a ConstantMedium (src/accel.rs:102-107, SURVEY Q12), and type 15 is the
// traversal's "leave instance" sentinel.
#define VKD_DUP 0x08000000u
#define VKD_INDEX(r) ((r)&0x07FFFFFFu)
#define VKD_TYPE(r) ((r) >> 28)
#define VKD_T_EXIT 15u
#define VKD_STACK 96

// Scene arrays in HBM.  Every record is a multiple of 16 B and fetched with 128-bit loads
// through the read-only path; one array per primitive kind (struct-of-arrays by type).
struct DScene {
    // Traversal layout: 4-wide nodes made from the reference's binary tree at upload (no rebuild: the
    // leaves, their boxes and therefore every closest hit are the reference's; only the grouping
    // changes).  A 4-wide node keeps the boxes of up to four descendants of one binary node -- its
    // children, with the larger inner children opened in turn -- so one visit (one 128-byte line,
    // eight independent 16-byte loads) decides four descents and halves the chain of dependent
    // memory round trips per ray.  Layout, 8 x float4 per binary node index (only the indices that
    // head a 4-wide node are filled):
    //   {min.x[4]} {max.x[4]} {min.y[4]} {max.y[4]} {min.z[4]} {max.z[4]} {ref[4]} {-}
    // A primitive slot carries the box of the binary node it hung under (the reference visits it only
    // when that box is hit); an empty slot has ref 0.
    const float4* wnodes;
    const float4* nodes;    // reference layout, 2 x float4 per node: {min.xyz, left}, {max.xyz, right}; used for
                            // the box of a BVH root (world root, instanced sub-BVH root)
    const float4* spheres;  // {center.xyz, radius}
    const uint32_t* sphere_mat;
    const float4* mspheres; // 3 x float4: {c0, r}, {c1, time0}, {time1, mat, -, -}
    const float4* rects;    // 2 x float4: {c0,c1,d0,d1}, {k, axes, mat, -}
    const float4* boxes;    // 2 x float4: {min.xyz, mat}, {max.xyz, -}
    const float4* xforms;   // 2 x float4: {kind, child, -, -}, {a, b, c, -}
    const float4* media;    // {boundary, neg_inv_density, mat, -}
    const float4* media_plan; // 4 x float4 per medium: the boundary's wrapper chain as one affine map + its leaf (Relayout::media_plan)
    const uint32_t* lights;
    const uint4* materials; // {type, tex, param, aux | needs_uv << 31}
    const uint4* textures;
    const uint8_t* texels;
    const float4* perlin_vec;   // 256 x float4 per Perlin
    const uint8_t* perlin_perm; // 768 B per Perlin (x, y, z)
    const float4* flat_shade;   // 2 x float4 per hit entry of the flat program (see Relayout::flat_shade); may be empty
    const uint8_t* prim_cls;    // shading class of every primitive (0 emitter, 1 dielectric, 2 metal, 3 the rest), one byte each:
    uint32_t cls_base[8];       // entry cls_base[type of the reference] + index of the reference (step-queue kernel's filing)
    uint32_t root;
    uint32_t n_lights;
    uint32_t has_media; // scene holds a ConstantMedium: selects the kernel instantiation with the medium code
    // A "simple" scene's one light, an unflipped Rect (Relayout::simple requires it): its record {c0,c1,d0,d1} {k, axes, mat, -}
    // once more in the kernel parameters, so that the trimmed build samples it from the constant bank (uniform loads, uniform
    // branches on its axes) instead of through lights[0] -> rects[] (three dependent loads per diffuse bounce and a per-lane
    // decode of the axes): Cornell 32.53 -> 31.14 ms, Cornell smoke 21.56 -> 21.08 ms.  The same shortcut as an extra
    // branch in the general builds LOSES (final scene 45.8 -> 48.9 ms, api demo 2.03 -> 2.30 ms: a second copy of the rect
    // code in kernels that are bound by instruction fetch; profiles/r2_sweep_18.log), so they do not have it.
    float4 light0_a, light0_b;
};
#define VKD_MAT_NEEDS_UV 0x80000000u

// ------------------------------------------------------------------------------------------------
// Flat traversal program.  A scene with few primitives (Cornell box: 13 rect sides + 1 sphere) gains
// nothing from its BVH on a GPU: the lanes of a warp sit at different nodes and execute each
// other's branches.  For such scenes vk_scene_upload unrolls the reference's traversal (a Boxy as
// its six sides, a wrapper chain as a change of ray frame) into typed, branch-free batches:
//
//   segment 0 = the world frame, segment s > 0 = one instance chain (its ops transform the world ray
//   into the object frame: Translate / RotateX,Y,Z, src/hittable.rs:508, :591-595, :680-684, :769-773);
//   inside a segment: XY rects, XZ rects, YZ rects (each kind once for plain rects and once for box
//   sides, which keep the list's strict `<` of src/hittable.rs:386), spheres, moving spheres, media.
//
// Every lane tests the SAME primitive at the same time with the SAME instruction sequence: no
// stack, no divergence, no type decode per entry, operands from the constant bank (the program
// travels as a __grid_constant__ kernel parameter).  Closest hit is order independent (exact ties
// excepted; a ConstantMedium's accept/reject does not depend on the tmax it is handed, only on
// whether a nearer surface exists), so this is the same function as BVHNode::hit.  The BVH path
// remains for everything larger.
// ------------------------------------------------------------------------------------------------
#define VKF_MAX_SEGS 12
#define VKF_MAX_OPS 24
#define VKF_MAX_RECTS 96
#define VKF_MAX_SPHERES 16
#define VKF_MAX_MEDIA 4
#define VKF_MAX_BVH 32
#define VKF_MAX_BOXES (VKF_MAX_RECTS / 6)
enum { VKF_OP_TRANSLATE = 0, VKF_OP_ROTX = 1, VKF_OP_ROTY = 2, VKF_OP_ROTZ = 3 };
struct FlatOp { // one wrapper level, outermost first
    uint32_t kind;
    float a, b, c; // translate: offset | rotate: sin, cos
};
struct FlatRect { // Rect::hit src/hittable.rs:230-239
    float4 bounds; // c0, c1, d0, d1
    float k;
    uint32_t hit;  // index into FlatProgram::hits
    uint32_t hitc; // the same index | queue class of the entry << 8 (VKF_HITC): what the K-ray trace returns
    uint32_t _pad;
};

struct FlatSphere { // Sphere::hit :65-95 | MovingSphere::hit :154-184
    float4 a; // center (center0), radius
    float4 b; // moving: center1, time0
    float time1;
    uint32_t hit;
    uint32_t hitc; // hit | queue class << 8
    uint32_t _pad;
};
// Queue class of a hit-table entry, carried in bits 8.. of the ids the K-ray trace returns (trace_flat_k), so that the
// warp-queue kernels file a traced ray without looking its entry up: 2 emitter, 3 dielectric, 4 metal, 5 diffuse,
// 6 diffuse behind an instance chain (the VKQ_* queue numbers of vk_warpq.cuh, asserted there).
#define VKF_HITC(index, cls, inst) ((uint32_t)(index) | (((cls) == 0u ? 2u : (cls) == 1u ? 3u : (cls) == 2u ? 4u : ((inst) ? 6u : 5u)) << 8))
#define VKF_HIT_INDEX(id) ((id)&0xFFu)
struct FlatBox { // Boxy::hit src/hittable.rs:363-365 as ONE entry (render build; the strict build tests its six sides as rects)
    float4 mn; // box_min, .w = bits: class-tagged id of side 0 (sides 0 and 1, the two XY rects, are consecutive entries)
    float4 mx; // box_max, .w = bits: class-tagged id of side 2 (XZ pair) | of side 4 (YZ pair) << 16
};
// A ConstantMedium entry of the flat program whose boundary is a Boxy (Cornell smoke), for the render build's K-ray trace:
// everything medium_t would fetch -- the medium record, its boundary chain as one affine map, the box -- in the constant
// bank, so the test runs inline on uniform operands (flat_medium_box).  flags 0: not such an entry, medium_t handles it.
struct FlatMedium {
    float aff[12]; // rows of R, then t: boundary frame = R * segment frame + t (identity without a chain)
    float4 mn;     // box_min, .w = -1 / density
    float4 mx;     // box_max, .w = bits: 1 = inline box entry | 2 = the boundary has a wrapper chain
};
struct FlatHit { // what the closest entry resolves to
    uint32_t prim; // leaf record (sphere / msphere / rect / box / medium [| VKD_DUP on a medium's second visit])
    uint32_t inst; // outermost wrapper of the chain it sits under, or 0
    uint32_t face; // box side 0..5 in Boxy::new order
    uint32_t cls;  // shading class of its material (VKW_* / VKS_C_*: 0 emitter, 1 dielectric, 2 metal, 3 diffuse)
};
struct FlatSeg {
    uint8_t op0, op1;           // ops [op0, op1) take the world ray into this segment's frame
    uint8_t rect0[6], rect1[6]; // rect ranges: XY, XZ, YZ plain, then XY, XZ, YZ box sides (strict)
    uint8_t sph0, sph1;         // static spheres
    uint8_t msph0, msph1;       // moving spheres
    uint8_t med0, med1;         // media: hits[] indices [med0, med1) (their prim is the medium ref)
    uint8_t bvh0, bvh1;         // sub-BVH roots [bvh0, bvh1) of FlatProgram::bvh, traversed in this segment's frame
    uint8_t box0, box1;         // boxes [box0, box1) of FlatProgram::boxes: the render build's form of the box-side rect ranges
};
struct FlatProgram {
    uint32_t n;      // number of primitive entries; 0 = no program: use the BVH
    uint32_t n_segs;
    uint32_t _pad[2];
    FlatSeg segs[VKF_MAX_SEGS];
    FlatOp ops[VKF_MAX_OPS];
    FlatRect rects[VKF_MAX_RECTS];
    FlatSphere spheres[VKF_MAX_SPHERES];
    FlatHit hits[VKF_MAX_RECTS + VKF_MAX_SPHERES + VKF_MAX_MEDIA];
    // Hybrid programs.  A heterogeneous scene (final scene: spheres, a moving sphere, media, a box field,
    // an instanced sphere cluster under one 13-node BVH) makes every lane of a warp test a different
    // KIND of primitive at the same time when it is traversed as a BVH (measured: 7.7 of 32 lanes
    // active, in the megakernel and in the dynamic-fetch wavefront extend alike).  The flat program
    // therefore unrolls only the heterogeneous top of the tree into typed batches and keeps each large
    // homogeneous subtree (all boxes, all spheres) as ONE entry: its root node, traversed through
    // the 4-wide nodes in the segment's frame, where every leaf test is the same code.
    uint32_t n_bvh;
    uint32_t bvh[VKF_MAX_BVH];           // node refs of the sub-BVH roots
    uint32_t seg_inst[VKF_MAX_SEGS];     // instance (outermost wrapper) of each segment, 0 for the world frame
    // The segment's chain of ops composed into one affine map (render build): object = R * world + t, rows of R then t.
    // The reference applies the wrappers one after the other (src/hittable.rs:508, :591-595); composing them on the host
    // changes the rounding only, so the strict build keeps walking the ops.
    float seg_affine[VKF_MAX_SEGS][12];
    // Render build: every Boxy of the program once more as one slab-test entry (flat_boxes_k, vk_device.cuh); it replaces the
    // box-side rect ranges rect0[3..5] there.  Same sides, same hit-table entries.
    FlatBox boxes[VKF_MAX_BOXES];
    FlatMedium fmed[VKF_MAX_MEDIA];
    uint8_t seg_fm0[VKF_MAX_SEGS]; // per segment: fmed entry of its first medium (entry i of hits[] is fmed[seg_fm0[s] + i - med0]);
                                   // kept out of FlatSeg: growing that record moves every array behind it in the constant bank,
                                   // which costs the Cornell kernel 0.5 % (31.15 -> 31.32 ms, profiles/r2_sweep_21.log)
};

// A flat program's SHAPE compiled into the warp-queue kernel (trace_flat_static, vk_device.cuh): per segment, the entry
// ranges the render build's trace reads -- rects per axis, static spheres, boxes -- as [begin, end) of FlatProgram's
// arrays.  The entries stay where the builder put them; the kernel reads them at constant offsets with every loop
// unrolled, instead of walking FlatSeg's byte ranges.  Every segment after the first is an instance frame with its affine
// map, as in trace_flat_k.  A program matches a shape when its segments read exactly these entries and nothing else (no
// moving sphere, medium or subtree).
template <int X0, int X1, int Y0, int Y1, int Z0, int Z1, int S0, int S1, int B0, int B1>
struct FlatSegShape {
    static constexpr int x0 = X0, x1 = X1, y0 = Y0, y1 = Y1, z0 = Z0, z1 = Z1, s0 = S0, s1 = S1, b0 = B0, b1 = B1;
    static bool matches(const FlatSeg& g) {
        auto same = [](uint32_t a0, uint32_t a1, int w0, int w1) { return a1 - a0 == (uint32_t)(w1 - w0) && (w1 == w0 || a0 == (uint32_t)w0); };
        return same(g.rect0[0], g.rect1[0], X0, X1) && same(g.rect0[1], g.rect1[1], Y0, Y1) && same(g.rect0[2], g.rect1[2], Z0, Z1) &&
               same(g.sph0, g.sph1, S0, S1) && same(g.box0, g.box1, B0, B1) && g.msph0 == g.msph1 && g.med0 == g.med1 && g.bvh0 == g.bvh1;
    }
};
template <class... Seg>
struct FlatShape {
    static constexpr uint32_t n_segs = sizeof...(Seg); // 0: no shape, the generic trace
    static bool matches(const FlatProgram& P) {
        uint32_t s = 0;
        return n_segs != 0 && P.n != 0 && P.n_segs == n_segs && P.n_bvh == 0 && (Seg::matches(P.segs[s++]) && ...);
    }
};
// The shapes the kernel is compiled for (vk_warpq.cu, namespace vkfast_simple), and the number naming each.
// cornell_box: the world frame (1 XY, 3 XZ, 2 YZ rects, the glass sphere), the rotated box's instance frame (one box)
using FlatShapeCornell = FlatShape<FlatSegShape<0, 1, 1, 4, 4, 6, 0, 1, 0, 0>, FlatSegShape<0, 0, 0, 0, 0, 0, 0, 0, 0, 1>>;
enum { VKF_SHAPE_NONE = 0, VKF_SHAPE_CORNELL = 1 };
inline uint32_t flat_static_shape(const FlatProgram& P) { return FlatShapeCornell::matches(P) ? (uint32_t)VKF_SHAPE_CORNELL : (uint32_t)VKF_SHAPE_NONE; }

struct DCamera {
    float3 origin, lower_left_corner, horizontal, vertical, u, v;
    float lens_radius, time0, time1;
};

struct RenderArgs {
    uint32_t width, height;
    uint32_t spp_begin, spp_count; // global sample range of this call
    uint32_t max_depth;
    uint32_t seed_lo, seed_hi;
    float3 background;
    uint32_t flags; // VK_FLAG_* of the call (sky background)
    // work decomposition of the lane megakernel (vk_api.cu decides): warp items = 8x4 pixel tiles x
    // chunks of chunk_spp samples; inside an item the lanes draw (pixel, sample) units
    uint32_t tiles_x, tiles_y, n_chunks, chunk_spp;
};

// Work domains: what the units of a render kernel run over.  Every kernel AUTO can pick takes its domain as its last
// template argument and as its last kernel parameter, behind all the others, so RenderArgs and everything in front of it
// keep one layout.  The bodies ask the domain the few questions of the "work domains" section of vk_device.cuh.
//   OneFrame   the W*H pixels of one frame (the single-frame kernels: the empty parameter adds nothing to their code)
//   FrameArgs  a batch of frames
//   ListArgs   a list of active pixels of one frame
//   FrameListArgs  a list of active pixels across a batch of frames
struct OneFrame {};

// A batch of frames (vk_render_frames): frame f renders with cams[f] and Philox key seed + f (64-bit add) into the
// accumulator plane that starts at f * n_pix * 3; pixel and sample of the Philox counter are the frame's own, so every frame
// equals its single-frame render.  The work units are frame-major (the frame is the outermost dimension): a warp whose
// frame has run dry takes the next frame's units, and the batch drains once.  Inside the warp-queue slots a pixel is the
// batch-wide index f * n_pix + y * width + x (the slot does not grow); the frame is recovered from it where a PathRng is
// rebuilt.
struct FrameArgs {
    const DCamera* cams; // device array, n_frames entries
    uint32_t n_frames;
    uint32_t n_pix;      // width * height
};

// A pass of an adaptive render (vk_render_adaptive): the work units run over a list of active pixels instead of the dense
// frame.  An entry is a frame pixel index y * width + x, so the accumulators keep their dense W*H*3 layout and a slot keeps
// the frame pixel.  Every kept sample also adds its per-channel square to `sq` (accumulate_square): 64-bit fixed point, so
// the sums, and the stopping decision made from them, do not depend on the order samples arrive in.
struct ListArgs {
    const uint32_t* list;   // active pixels, ascending
    uint32_t n;             // list length
    unsigned long long* sq; // W*H*3 fixed-point sums of squares (VK_SQ_SCALE)
};

// A pass of an adaptive render of a batch of frames (vk_render_frames_adaptive): one list of active pixels across all the
// frames.  An entry is the batch-wide pixel g = f * n_pix + y * width + x, ascending, so it is the index of the batch's
// contiguous accumulator planes (and of the squares, ls.sq: n_frames * W*H*3) and what a warp-queue slot keeps in a batch.
// Each unit resolves its own frame from g: the camera fr.cams[f], the key seed + f and the frame pixel g - f * n_pix, so every
// frame equals its single-frame adaptive render.  The units run over the list alone (fr.n_frames does not multiply them).
struct FrameListArgs {
    FrameArgs fr;
    ListArgs ls;
};
// Squares: VK_SQ_SCALE = 2^32 units per 1.0, each channel of a sample clamped to VK_SQ_CLAMP before it is squared (the clamp
// touches the statistic only, never the image).  One sample adds at most 255^2 * 2^32 < 2^48 units, so VK_ADAPTIVE_MAX_SPP =
// 2^16 samples stay below 2^64.
#define VK_SQ_SCALE 4294967296.0f
#define VK_SQ_INV_SCALE (1.0 / 4294967296.0)
#define VK_SQ_CLAMP 255.0f
#define VK_ADAPTIVE_MAX_SPP 65536u

// Accumulation.  Every finished sample is added to its pixel with three 64-bit integer atomics
// (fixed point, VK_ACC_SCALE = 2^30 units per 1.0): integer addition is associative, so the frame is
// bit-identical for a (seed, sample range, image size) whatever the kernel variant, the scheduling of
// paths onto lanes, the grid or the number of GPUs that rendered other sample ranges -- and no lane
// has to own a pixel's samples in order (round 1 spent one fp32 plane per sample, 4.3 GB per Cornell
// frame, to get the same property).  Range +-2^33 per pixel and channel, resolution 9.3e-10; a sample
// is clamped to +-2^32 before conversion.  The sums of squares (tests only) are double atomics.
// counters[0] = rays, [1] = dropped samples, [2] = work-queue head, [3] = node visits, [4] = primitive tests
#define VK_ACC_SCALE 1073741824.0f
#define VK_ACC_INV_SCALE (1.0 / 1073741824.0)
struct RenderBuffers {
    unsigned long long* acc; // W*H*3 fixed-point sums (two's complement)
    double* accsq;           // W*H*3 sums of squares, nullable
    unsigned long long* counters;
    unsigned long long* debug; // VK_DEBUG_CTAS x {end time ns, rays traced, smid, -} of the staged kernel's CTAs
};
#define VK_DEBUG_CTAS 2048

// ------------------------------------------------------------------------------------------------
// Wavefront variant: a pool of path slots in device memory (L2-resident at the default pool size),
// advanced one segment per iteration by separate kernels:
//   generate  k_wf_generate  every slot takes a (pixel, sample block) unit and its first camera ray
//   extend    k_wf_extend    world.hit() for every live slot; the hit is classified by the material's
//                            shading class and the slot index appended to that class's queue
//                            (warp ballot + one atomic per warp and class)
//   shade     k_wf_shade     walks the queues class by class, so a warp shades one kind of material:
//                            scatter + PDF sampling, or sample end -> accumulate -> next sample / next
//                            unit (regeneration in place: the pool stays full until units run out)
// A finished sample goes into its pixel's integer accumulators, exactly like a lane of the megakernel:
// both variants produce the same image for a seed.  float4 / uint4 arrays: every access is one fully
// coalesced 16 B per lane.
// ------------------------------------------------------------------------------------------------
enum { VKW_TERMINATE = 0, VKW_DIELECTRIC = 1, VKW_METAL = 2, VKW_DIFFUSE = 3, VKW_CLASSES = 4 };
struct WfState {
    float4* ray_o;  // origin.xyz, time
    float4* ray_d;  // direction.xyz, bits: depth of the segment to trace (0 = slot idle)
    float4* beta;   // path weight.xyz, bits: global index of the current sample
    uint4* unit;    // pixel, -, -, -
    uint4* hit;     // t bits, primitive, instance, face
    uint32_t* queue;    // VKW_CLASSES x n_slots slot indices
    uint32_t* qcount;   // 2 sets x VKW_CLASSES counters (set = iteration parity)
    unsigned long long* unit_head; // next unit to hand out
    uint32_t n_slots;
    uint32_t n_pixels;
    unsigned long long n_units;
};

// (the launchers that take a work domain D are instantiated for OneFrame, FrameArgs, ListArgs and FrameListArgs)
#define VK_DECLARE_LAUNCHERS(NS)                                                                                       \
    namespace NS {                                                                                                     \
    template <class D>                                                                                                 \
    cudaError_t launch_megakernel(const DScene& sc, const FlatProgram* flat, const DCamera& cam, const RenderArgs& a,  \
                                  const RenderBuffers& b, int grid, bool legacy, cudaStream_t st, const D& dom);       \
    template <class D>                                                                                                 \
    cudaError_t launch_megakernel_dyn(const DScene& sc, const DCamera& cam, const RenderArgs& a, const RenderBuffers& b, \
                                      unsigned long long* unit_head, int sm_count, cudaStream_t st, const D& dom);     \
    cudaError_t launch_intersect(const DScene& sc, const FlatProgram* flat, const vk_ray* rays, size_t n,              \
                                 const float* medium_xi, vk_hit* out, cudaStream_t st);                                \
    cudaError_t megakernel_occupancy(bool flat, bool media, bool legacy, int* blocks_per_sm, int* block_threads);      \
    cudaError_t launch_philox_kat(const uint32_t* ctr_key6, uint32_t* out4, cudaStream_t st);                          \
    cudaError_t launch_eval(const DScene& sc, vk_eval* recs, size_t n, uint32_t n_materials, uint32_t n_textures,      \
                            cudaStream_t st);                                                                          \
    cudaError_t launch_staged(const DScene& sc, const FlatProgram* flat, const DCamera& cam, const RenderArgs& a,      \
                              const RenderBuffers& b, unsigned long long* unit_head, int sm_count, cudaStream_t st);   \
    template <class D>                                                                                                 \
    cudaError_t launch_warpq(const DScene& sc, const FlatProgram* flat, uint32_t flat_shape, const DCamera& cam,       \
                             const RenderArgs& a, const RenderBuffers& b, unsigned long long* unit_head, int sm_count, \
                             bool legacy, cudaStream_t st, const D& dom);                                              \
    size_t stepq_stack_words(uint32_t stack_need, bool inst, int sm_count, uint32_t* levels);                          \
    template <class D>                                                                                                 \
    cudaError_t launch_stepq(const DScene& sc, const DCamera& cam, const RenderArgs& a, const RenderBuffers& b,        \
                             unsigned long long* unit_head, uint32_t* gstack, uint32_t glevels, bool inst, int sm_count, \
                             bool legacy, cudaStream_t st, const D& dom);                                              \
    cudaError_t launch_wf_generate(const DCamera& cam, const RenderArgs& a, const WfState& w, cudaStream_t st);        \
    cudaError_t launch_wf_extend(const DScene& sc, const FlatProgram* flat, const RenderArgs& a, const WfState& w,     \
                                 const RenderBuffers& b, uint32_t set, cudaStream_t st);                               \
    cudaError_t launch_wf_shade(const DScene& sc, const DCamera& cam, const RenderArgs& a, const WfState& w,           \
                                const RenderBuffers& b, uint32_t set, cudaStream_t st);                                \
    }
VK_DECLARE_LAUNCHERS(vkfast)
VK_DECLARE_LAUNCHERS(vkstrict)
VK_DECLARE_LAUNCHERS(vkfast_l0) // (vk_kernels.cu, vk_warpq.cu, vk_stepq.cu with VK_LIGHT0=1: the megakernel, warp-queue and step-queue launchers only)
// vk_render_aov's kernel (vk_kernels.cu), in the render and strict builds: the feature planes of n_frames frames (cams: device
// array; a.tiles_x x a.tiles_y: one frame's 8x4 tiles) written whole into the nullable device planes; use_flat: traverse
// `flat`, otherwise the BVH.  counters[0] / [3] / [4]: rays, node visits, primitive tests.
#define VK_DECLARE_AOV(NS)                                                                                             \
    namespace NS {                                                                                                     \
    cudaError_t launch_aov(const DScene& sc, const FlatProgram& flat, bool use_flat, const DCamera* cams, uint32_t n_frames, \
                           const RenderArgs& a, uint32_t aov_spp, float* albedo, float* normal, float* depth, float* coverage, \
                           unsigned long long* counters, cudaStream_t st);                                             \
    }
VK_DECLARE_AOV(vkfast)
VK_DECLARE_AOV(vkstrict)
namespace vkfast_simple { // vk_staged.cu / vk_warpq.cu compiled with VK_SIMPLE=1: kernels for "simple" flat scenes (see vk_device.cuh)
cudaError_t launch_staged(const DScene& sc, const FlatProgram* flat, const DCamera& cam, const RenderArgs& a, const RenderBuffers& b,
                          unsigned long long* unit_head, int sm_count, cudaStream_t st);
template <class D>
cudaError_t launch_warpq(const DScene& sc, const FlatProgram* flat, uint32_t flat_shape, const DCamera& cam, const RenderArgs& a,
                         const RenderBuffers& b, unsigned long long* unit_head, int sm_count, bool legacy, cudaStream_t st, const D& dom);
}
