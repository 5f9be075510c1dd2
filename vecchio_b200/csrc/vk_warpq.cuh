// vk_warpq.cuh -- what the warp-queue kernels share (vk_warpq.cu: flat programs and the lane-traversal BVH kernel;
// vk_stepq.cu: the BVH kernel with one queue per traversal step): slot pool, rings, unit regeneration, the shade batch.
#pragma once
#include "vk_device.cuh"

namespace VK_NS {

// Per kernel family (measured on B200, profiles/r2_sweep_*.log):
//   flat program, no medium   176 slots, 2 rays per lane in extend, 4 CTAs x 4 warps per SM: the extend's instruction-
//                             level parallelism and a pool deep enough that every batch is full matter, more warps do not
//                             (24 warps x 120 slots: 43.0 against 40.0 ms per Cornell frame; 1 / 3 rays per lane: 47.4 / 38.9)
//   flat program with media   120 slots, 1 ray per lane, 6 CTAs per SM: the medium test is a call per ray with a Philox
//                             block and a logf behind it -- latency, not issue -- and wants the warps (Cornell smoke, 500 spp:
//                             26.9 ms against 30.9 with the first configuration and 36.3 for the CTA-staged kernel)
//   BVH                       120 slots, 6 CTAs per SM (traversal is memory latency: 63.8 against 65.5 ms on the final scene,
//                             37.6 against 48.6 on 10^6 spheres)
// A slot is 68 B; rings hold slot indices as bytes (capacity a power of two >= slots); 16 x (68 x 176 + 7 x 256) and
// 24 x (68 x 120 + 7 x 128) both come to 220 KB of the SM's 227 KB of shared memory.
#ifndef VKQ_WARPS
#define VKQ_WARPS 4
#endif
#ifndef VKQ_N_FLAT
#define VKQ_N_FLAT 176
#endif
#ifndef VKQ_RN_FLAT
#define VKQ_RN_FLAT 256
#endif
#ifndef VKQ_K_FLAT
#define VKQ_K_FLAT 2
#endif
#ifndef VKQ_MINB_FLAT
#define VKQ_MINB_FLAT 4
#endif
#ifndef VKQ_N_MEDIA
#define VKQ_N_MEDIA 144
#endif
#ifndef VKQ_RN_MEDIA
#define VKQ_RN_MEDIA 256
#endif
#ifndef VKQ_K_MEDIA
#define VKQ_K_MEDIA 1
#endif
#ifndef VKQ_MINB_MEDIA
#define VKQ_MINB_MEDIA 5
#endif
#ifndef VKQ_N_BVH
#define VKQ_N_BVH 120
#endif
#ifndef VKQ_RN_BVH
#define VKQ_RN_BVH 128
#endif
#ifndef VKQ_MINB_BVH
#define VKQ_MINB_BVH 6
#endif
// hybrid programs (flat top + homogeneous subtrees walked inside extend): the BVH family's shape
#ifndef VKQ_N_HYB
#define VKQ_N_HYB 120
#endif
#ifndef VKQ_RN_HYB
#define VKQ_RN_HYB 128
#endif
#ifndef VKQ_MINB_HYB
#define VKQ_MINB_HYB 6
#endif
#ifndef VKQ_REGEN_MIN
#define VKQ_REGEN_MIN 32u // ended lanes of a shade batch are regenerated at once when at least this many ended (8 / 16 / 32:
                          // Cornell 31.34 / 31.20 / 31.13 ms, smoke 18.54 / 18.47 / 18.42 ms, profiles/r2_sweep_23.log)
#endif
#define VKQ_CHUNK 256u
// (7 .. 9: the traversal-step queues of vk_stepq.cu, where VKQ_EXT holds the rays whose next step is a node visit)
enum { VKQ_EXT = 0, VKQ_END = 1, VKQ_EMIT = 2, VKQ_DIEL = 3, VKQ_METAL = 4, VKQ_DIFF = 5, VKQ_DIFFI = 6, VKQ_NQ = 7,
       VKQ_SPH = 7, VKQ_BOX = 8, VKQ_LEAF = 9, VKQ_NQ_STEP = 10, VKQ_NONE = 15 };
static_assert(VKF_HITC(0, 0, 0) >> 8 == VKQ_EMIT && VKF_HITC(0, 1, 0) >> 8 == VKQ_DIEL && VKF_HITC(0, 2, 0) >> 8 == VKQ_METAL &&
              VKF_HITC(0, 3, 0) >> 8 == VKQ_DIFF && VKF_HITC(0, 3, 1) >> 8 == VKQ_DIFFI, "the flat program's class-tagged ids name these queues");

template <int N_, int RN_>
struct WqWarp {
    static constexpr uint32_t N = N_, RMASK = RN_ - 1, NQ = VKQ_NQ;
    static_assert((RN_ & (RN_ - 1)) == 0 && RN_ >= N_ && RN_ <= 256, "ring capacity: power of two, >= slots, byte indices");
    float4 ro[N_];            // origin.xyz, time
    float4 rd[N_];            // direction.xyz, bits: depth of the segment to trace
    float4 bt[N_];            // path weight.xyz, bits: global sample index
    uint4 hp[N_];             // hit: t bits, primitive, instance index | face << 28 | has-instance << 31; flat hit entry
    uint32_t px[N_];          // pixel of the slot's sample
    uint8_t ring[VKQ_NQ][RN_]; // slot indices, one ring per queue
    uint2 ct[8];                 // per queue: .x = entries, .y = ring write position
    uint32_t cur_s, cur_y, cur_x, left; // unit cursor: next unit is (sample cur_s, row cur_y, column cur_x); `left` units remain in the chunk
    uint32_t exhausted;          // the global unit counter has run past the end
    VKD void mark_new(uint32_t) {} // (a new ray segment was written to the slot: nothing else to reset here)
};


// A barrier of the warp with itself (named barrier 1 + warp index, 32 threads).  Functionally a __syncwarp; what it buys
// is in the compiler: ptxas only uses the uniform datapath (uniform loop counters, LDCU constant loads, BRA.U) in code
// it can prove the whole warp executes together, and inside this kernel's scheduler loop it cannot -- after an ALIGNED
// barrier it can.  Without it the flat program's operands are fetched with per-thread indexed constant loads
// (measured in SASS: 37 -> 77 uniform loads, all six rect loops on the uniform datapath).
#ifndef VKQ_CONVERGE
#define VKQ_CONVERGE 1
#endif
VKD void wq_converge() {
#if VKQ_CONVERGE
    asm volatile("barrier.sync.aligned %0, 32;" ::"r"((threadIdx.x >> 5) + 1u) : "memory");
#endif
}
// (the work domain travels beside the context, as an argument of its own: as a reference member it changed the code of
// the single-frame kernels, whose domain is empty)
template <class W>
struct WqCtx {
    const DCamera& cam;
    const RenderArgs& a;
    W& S;
    uint32_t chunks_per_row, chunks_per_sample; // a chunk: up to VKQ_CHUNK consecutive pixels of one row of one sample
    unsigned long long n_chunks;
    unsigned long long* unit_head;
    uint32_t lane, below;
};

// ---- the work domains' chunks (see vk_device.cuh) ---------------------------------------------------------------------
// One frame: chunk c = (sample * height + row) * chunks_per_row + segment.  A batch: the same, frame-major, and the unit
// cursor's row is then the batch-wide row f * height + y.  A list: VKQ_CHUNK consecutive entries of one sample (the list is
// one row), and the cursor's column is then a list index.
template <class D> VKD uint32_t wq_row_length(const D&, const RenderArgs& a) { return a.width; }
VKD uint32_t wq_row_length(const ListArgs& ls, const RenderArgs&) { return ls.n; }
VKD uint32_t wq_row_length(const FrameListArgs& fl, const RenderArgs&) { return fl.ls.n; }
template <class D> VKD uint32_t wq_rows(const D&, const RenderArgs& a) { return a.height; }
VKD uint32_t wq_rows(const ListArgs&, const RenderArgs&) { return 1u; }
VKD uint32_t wq_rows(const FrameListArgs&, const RenderArgs&) { return 1u; }
template <class W, class D>
VKD WqCtx<W> wq_ctx(const D& dom, const DCamera& cam, const RenderArgs& a, W& S, unsigned long long* unit_head, uint32_t lane) {
    const uint32_t cpr = (wq_row_length(dom, a) + VKQ_CHUNK - 1u) / VKQ_CHUNK, cps = cpr * wq_rows(dom, a);
    return WqCtx<W>{cam, a, S, cpr, cps, (unsigned long long)cps * a.spp_count * dom_frames(dom), unit_head, lane, (1u << lane) - 1u};
}
// chunk c -> the unit cursor of the warp (lane 0 only)
template <class W>
VKD void wq_chunk(const WqCtx<W>& C, const OneFrame&, unsigned long long c) {
    W& S = C.S;
    const uint32_t sb = (uint32_t)(c / C.chunks_per_sample);
    const uint32_t r = (uint32_t)(c - (unsigned long long)sb * C.chunks_per_sample);
    const uint32_t row = r / C.chunks_per_row, x0 = (r - row * C.chunks_per_row) * VKQ_CHUNK;
    S.left = min(VKQ_CHUNK, C.a.width - x0);
    S.cur_s = sb;
    S.cur_y = row;
    S.cur_x = x0;
}
template <class W>
VKD void wq_chunk(const WqCtx<W>& C, const FrameArgs&, unsigned long long c) {
    // c = ((f * spp_count + sample) * height + row) * chunks_per_row + segment; f * spp_count + sample stays 64-bit until
    // the frame is split off (it passes 2^32 long before the batch's pixel index does)
    W& S = C.S;
    const unsigned long long fs = c / C.chunks_per_sample;
    const uint32_t f = (uint32_t)(fs / C.a.spp_count);
    const uint32_t r = (uint32_t)(c - fs * C.chunks_per_sample);
    const uint32_t row = r / C.chunks_per_row, x0 = (r - row * C.chunks_per_row) * VKQ_CHUNK;
    S.left = min(VKQ_CHUNK, C.a.width - x0);
    S.cur_s = (uint32_t)(fs - (unsigned long long)f * C.a.spp_count);
    S.cur_y = f * C.a.height + row;
    S.cur_x = x0;
}
template <class W>
VKD void wq_chunk(const WqCtx<W>& C, const ListArgs& ls, unsigned long long c) { // c = sample * chunks_per_sample + chunk of the list
    W& S = C.S;
    const uint32_t sb = (uint32_t)(c / C.chunks_per_sample);
    const uint32_t x0 = ((uint32_t)c - sb * C.chunks_per_sample) * VKQ_CHUNK;
    S.left = min(VKQ_CHUNK, ls.n - x0);
    S.cur_s = sb;
    S.cur_y = 0u;
    S.cur_x = x0;
}
template <class W>
VKD void wq_chunk(const WqCtx<W>& C, const FrameListArgs& fl, unsigned long long c) { wq_chunk(C, fl.ls, c); } // (a list is a list)
// The unit (x, y) of the cursor, rng.pixel = y * width + x: the camera ray of the pixel it stands for, with that pixel's
// Philox counter pixel and key.  Returns the pixel the slot keeps: the accumulator index.
template <class W>
VKD uint32_t wq_camera_ray(const WqCtx<W>& C, const OneFrame&, uint32_t x, uint32_t y, PathRng& rng, float3& o, float3& d, float& time) {
    camera_get_ray(C.cam, rng, x, y, C.a.width, C.a.height, o, d, time);
    return rng.pixel;
}
template <class W>
VKD uint32_t wq_camera_ray(const WqCtx<W>& C, const FrameArgs& fr, uint32_t x, uint32_t y, PathRng& rng, float3& o, float3& d, float& time) {
    const uint32_t p = rng.pixel; // y is the batch-wide row, p the batch-wide pixel
    const uint32_t f = y / C.a.height;
    y -= f * C.a.height;
    rng.pixel = y * C.a.width + x;
    rng.key = frame_key(C.a, f);
    camera_get_ray(fr.cams[f], rng, x, y, C.a.width, C.a.height, o, d, time);
    return p;
}
template <class W>
VKD uint32_t wq_camera_ray(const WqCtx<W>& C, const ListArgs& ls, uint32_t x, uint32_t y, PathRng& rng, float3& o, float3& d, float& time) {
    rng.pixel = ls.list[x]; // x is a list index
    y = rng.pixel / C.a.width;
    x = rng.pixel - y * C.a.width;
    camera_get_ray(C.cam, rng, x, y, C.a.width, C.a.height, o, d, time);
    return rng.pixel;
}
template <class W>
VKD uint32_t wq_camera_ray(const WqCtx<W>& C, const FrameListArgs& fl, uint32_t x, uint32_t, PathRng& rng, float3& o, float3& d, float& time) {
    const uint32_t g = fl.ls.list[x]; // x is a list index, the entry a batch-wide pixel
    rng.pixel = g;
    const uint32_t f = dom_unit_frame(fl, C.a, rng);
    const uint32_t y = rng.pixel / C.a.width;
    camera_get_ray(fl.fr.cams[f], rng, rng.pixel - y * C.a.width, y, C.a.width, C.a.height, o, d, time);
    return g;
}

// Append the lanes with cls != VKQ_NONE to the queue of their class: one match groups the lanes, the first
// lane of each group moves that queue's counters (no other lane touches them: different groups, different queues).
template <class W>
VKD void wq_push(W& S, uint32_t cls, uint32_t slot, uint32_t lane, uint32_t below) {
    const uint32_t m = __match_any_sync(0xFFFFFFFFu, cls);
    const uint32_t leader = __ffs(m) - 1u;
    uint32_t pos = 0;
    if (lane == leader && cls != VKQ_NONE) {
        const uint2 c = S.ct[cls];
        pos = c.y;
        S.ct[cls] = make_uint2(c.x + (uint32_t)__popc(m), c.y + (uint32_t)__popc(m));
    }
    pos = __shfl_sync(0xFFFFFFFFu, pos, leader);
    if (cls != VKQ_NONE) S.ring[cls][(pos + __popc(m & below)) & W::RMASK] = (uint8_t)slot;
    __syncwarp();
}

// The lanes with want == true take the warp's next units and start their camera ray (src/main.rs:187-190).
// Returns whether this lane got one (false: the frame has no unit left, the slot retires).
// Units are dealt in CHUNKS from one global counter: a chunk is up to VKQ_CHUNK consecutive pixels of ONE row of ONE
// sample, so the lanes' units are (s, y, x0 + i) with nothing to wrap and nothing to divide; lane 0 splits the chunk
// number into (sample, row, row segment) once per chunk.  Which warp renders which unit does not show in the image
// (Philox is keyed by pixel and sample, the accumulators are integers).
template <class W, class D>
VKD bool wq_regen(const WqCtx<W>& C, const D& dom, bool want, uint32_t slot) {
    W& S = C.S;
    const uint32_t m = __ballot_sync(0xFFFFFFFFu, want);
    if (m == 0u) return false;
    const uint32_t need = (uint32_t)__popc(m), rank = (uint32_t)__popc(m & C.below);
    uint32_t served = 0, s = 0, y = 0, x = 0;
    bool got = false;
#pragma unroll 1
    while (served < need) { // at most two rounds: what the current chunk still holds, then a new chunk
        // (the warp reductions / votes only make values every lane already agrees on PROVABLY uniform: __syncwarp
        // under a branch the compiler must assume divergent costs the whole kernel its uniform-datapath code)
        uint32_t left = __reduce_max_sync(0xFFFFFFFFu, S.left);
        if (left == 0u) {
            if (__any_sync(0xFFFFFFFFu, S.exhausted != 0u)) break;
            __syncwarp();
            if (C.lane == 0) {
                const unsigned long long c = atomicAdd(C.unit_head, 1ull);
                if (c >= C.n_chunks) S.exhausted = 1u;
                else wq_chunk(C, dom, c);
            }
            __syncwarp();
            if (__any_sync(0xFFFFFFFFu, S.exhausted != 0u)) break;
            left = __reduce_max_sync(0xFFFFFFFFu, S.left);
        }
        const uint32_t take = min(need - served, left);
        const uint32_t cs = S.cur_s, cy = S.cur_y, cx = S.cur_x;
        if (want && rank >= served && rank < served + take) {
            x = cx + (rank - served);
            y = cy;
            s = cs;
            got = true;
        }
        __syncwarp();
        if (C.lane == 0) {
            S.cur_x = cx + take;
            S.left = left - take;
        }
        __syncwarp();
        served += take;
    }
    if (got) {
        PathRng rng;
        rng.pixel = y * C.a.width + x; // i = y*width + x, row 0 = bottom (src/main.rs:182-183)
        rng.sample = C.a.spp_begin + s;
        rng.key = make_uint2(C.a.seed_lo, C.a.seed_hi);
        float3 o, d;
        float time;
        const uint32_t p = wq_camera_ray(C, dom, x, y, rng, o, d, time);
        S.ro[slot] = make_float4(o.x, o.y, o.z, time);
        S.rd[slot] = make_float4(d.x, d.y, d.z, __uint_as_float(1u)); // ray_color(ray, .., 1)
        S.bt[slot] = make_float4(1.0f, 1.0f, 1.0f, __uint_as_float(rng.sample));
        S.px[slot] = p;
        S.mark_new(slot);
    }
    return got;
}

VKD bool wq_black_miss(const RenderArgs& a) {
    return !(a.flags & VK_FLAG_SKY_BACKGROUND) && a.background.x == 0.0f && a.background.y == 0.0f && a.background.z == 0.0f;
}
VKD uint32_t wq_class_of(const DScene& sc, uint32_t prim, uint32_t inst) {
    uint32_t mat;
    const uint32_t i = VKD_INDEX(prim);
    switch (VKD_TYPE(prim)) {
    case VK_T_SPHERE: mat = __ldg(&sc.sphere_mat[i]); break;
    case VK_T_MSPHERE: mat = __float_as_uint(__ldg(&sc.mspheres[3 * i + 2]).y); break;
    case VK_T_RECT: mat = __float_as_uint(__ldg(&sc.rects[2 * i + 1]).z); break;
    case VK_T_BOX: mat = __float_as_uint(__ldg(&sc.boxes[2 * i]).w); break;
    default: mat = __float_as_uint(__ldg(&sc.media[i]).z); break;
    }
    const uint32_t t = __ldg(&sc.materials[mat]).x;
    return t == VK_M_DIFFUSE_LIGHT ? VKQ_EMIT : t == VK_M_DIELECTRIC ? VKQ_DIEL : t == VK_M_METAL ? VKQ_METAL : (inst ? VKQ_DIFFI : VKQ_DIFF);
}

// Queue counters of the warp: {entries, ring write position} per queue.
struct WqCounts {
    uint4 c01, c23, c45, c67; // EXT END | EMIT DIEL | METAL DIFF | DIFFI -
};
template <class W>
VKD WqCounts wq_counts(const W& S) {
    WqCounts c;
    c.c01 = *reinterpret_cast<const uint4*>(&S.ct[0]);
    c.c23 = *reinterpret_cast<const uint4*>(&S.ct[2]);
    c.c45 = *reinterpret_cast<const uint4*>(&S.ct[4]);
    c.c67 = *reinterpret_cast<const uint4*>(&S.ct[6]);
    return c;
}
// The fullest queue: score = entries / batch width (EXT batches are ext_cap wide, the others 32; ext_cap == 0 leaves
// the extend queue out).  Returns false when every considered queue is empty.  One max chain over (score << 3 | queue).
template <class W>
VKD bool wq_pick(const W& S, const WqCounts& c, uint32_t ext_cap, uint32_t& q, uint32_t& n_q, uint32_t& tail_q) {
    const uint32_t w = (ext_cap ? ext_cap : 32u) * 8u;
    uint32_t key = ext_cap ? c.c01.x * 256u + VKQ_EXT : 0u; // entries * 32 * 8 | queue
    key = max(key, c.c23.x * w + VKQ_EMIT);
    key = max(key, c.c45.z * w + VKQ_DIFF);
    key = max(key, c.c67.x * w + VKQ_DIFFI);
    key = max(key, c.c23.z * w + VKQ_DIEL);
    key = max(key, c.c45.x * w + VKQ_METAL);
    key = max(key, c.c01.z * w + VKQ_END);
    // Every lane computed the same value from the same shared-memory words, but the compiler cannot know that: a
    // warp reduction (REDUX, result in a uniform register) makes the choice provably warp-uniform, so the stage it
    // selects runs under uniform control flow (uniform-datapath loop counters and constant loads in the traversal).
    key = __reduce_max_sync(0xFFFFFFFFu, key);
    q = key & 7u;
    const uint2 e = S.ct[q];
    n_q = e.x;
    tail_q = e.y;
    return (key >> 3) != 0u;
}
// Take up to `cap` entries off queue q: returns how many, and the ring position of the first.
template <class W>
VKD uint32_t wq_pop(W& S, uint32_t q, uint32_t n_q, uint32_t tail_q, uint32_t cap, uint32_t lane, uint32_t& head) {
    const uint32_t n = min(n_q, cap);
    head = tail_q - n_q;
    __syncwarp();
    if (lane == 0) S.ct[q].x = n_q - n;
    __syncwarp();
    // (the entries [head, head + n) stay readable: pushes only write at the ring's tail, and a ring holds at least as many entries as the warp has slots)
    return n;
}

// One batch of a shading class (or of the regeneration queue): resolve + scatter (src/main.rs:131-149); a finished sample
// goes through the NaN / Inf filter (:191-194) into its pixel; survivors go to the extend queue.
// VKQ_FAST_RESOLVE (render build, flat scenes): a rect / box-side hit whose HitRec can be written down directly
// (DScene::flat_shade, decided at upload) skips resolve_hit's walk down and up the wrapper chain: p = o + t d in the
// world frame, normal = the entry's constant world normal turned against the ray.
#ifndef VKQ_FAST_RESOLVE
#define VKQ_FAST_RESOLVE 1 // (Cornell, 1000 spp: 37.9 against 40.0 ms per frame)
#endif
// The shading of one lane's slot (act: the lane holds one), in the batch of a class.  CLS: the class every slot of the
// batch has -- VKQ_EMIT (emitters and misses), VKQ_DIEL, VKQ_DIFF (Lambertian / Isotropic, the DIFF and DIFFI queues
// alike) -- so that the code is that class's shading body alone; VKQ_NQ: any class, shade_xi's dispatch on the material.
// The queue a slot sits in comes from its material at upload (VKF_HITC), so a slot of another class cannot occur: the
// VKQ_SELFCHECK build counts one as a violation.
template <bool LEGACY, bool FLAT, int CLS, class W, class D>
VKD void wq_shade_slot(const DScene& sc, const WqCtx<W>& C, const D& dom, const RenderBuffers& buf, bool act, uint32_t slot, bool& alive,
                       bool& ended, uint32_t& n_drop) {
    static_assert(CLS == VKQ_NQ || (!LEGACY && (CLS == VKQ_EMIT || CLS == VKQ_DIEL || CLS == VKQ_DIFF)),
                  "class bodies: the HEAD integrator's emitter, dielectric and diffuse");
    W& S = C.S;
    const RenderArgs& a = C.a;
    if (act) {
        const float4 ro = S.ro[slot], rd = S.rd[slot], bt = S.bt[slot];
        const uint4 hp = S.hp[slot];
        float3 o = f3(ro), d = f3(rd), beta = f3(bt), L = f3(0.0f, 0.0f, 0.0f);
        float time = ro.w;
        uint32_t depth = __float_as_uint(rd.w);
        const uint32_t pixel = S.px[slot], prim = hp.y;
        bool valid = true;
#if VKQ_SELFCHECK
        if (CLS != VKQ_NQ && CLS != VKQ_EMIT && prim == VK_REF_NONE) atomicAdd(&buf.counters[5], 1ull); // (a miss files as an emitter)
#endif
        if ((CLS == VKQ_NQ || CLS == VKQ_EMIT) && prim == VK_REF_NONE) {
            L = beta * miss_color(a, d); // src/main.rs:151
        } else {
            PathRng rng;
            rng.pixel = pixel;
            rng.sample = __float_as_uint(bt.w);
            rng.key = make_uint2(a.seed_lo, a.seed_hi);
            dom_slot_rng(dom, a, rng); // (the slot's pixel is the accumulator index: batch-wide in a batch)
            HitRecD rec;
            bool direct = false;
            uint32_t leaf = prim, hi = hp.z;
            if (FLAT) { // a flat program's slot keeps the distance and the hit-table entry; the rest hangs under the entry
                const float4 fs1 = __ldg(&sc.flat_shade[2u * hp.w + 1u]);
                leaf = __float_as_uint(fs1.y);
                hi = __float_as_uint(fs1.z);
#if VKQ_FAST_RESOLVE && !VK_STRICT
                const float4 fs = __ldg(&sc.flat_shade[2u * hp.w]);
                const uint32_t fl = __float_as_uint(fs.w);
                if (fl & 1u) {
                    direct = true;
                    const float3 nw = f3(fs);
                    const bool toward = dot3(d, nw) < 0.0f;
                    rec.t = __uint_as_float(hp.x);
                    rec.p = at(o, d, rec.t);
                    rec.normal = toward ? nw : -nw;
                    rec.front = (toward ? 1u : 0u) ^ ((fl >> 1) & 1u);
                    rec.u = 0.0f;
                    rec.v = 0.0f;
                    rec.mat = __float_as_uint(fs1.x);
                    rec.m = __ldg(&sc.materials[rec.mat]);
                }
#endif
            }
            if (!direct) {
                TraceHit h;
                h.t = __uint_as_float(hp.x);
                h.prim = leaf;
                h.inst = (hi & 0x80000000u) ? (((uint32_t)VK_T_XFORM << 28) | (hi & 0x07FFFFFFu)) : 0u;
                h.face = (hi >> 28) & 7u;
                resolve_hit(sc, h, o, d, time, false, rec);
            }
            if constexpr (CLS == VKQ_NQ) {
                alive = LEGACY ? shade_legacy(sc, rec, rng, depth, o, d, time, beta, L, valid)
                               : shade(sc, rec, rng, depth, o, d, time, beta, L, valid);
            } else {
#if VKQ_SELFCHECK
                const uint32_t t = rec.m.x;
                const uint32_t mc = t == VK_M_DIFFUSE_LIGHT ? VKQ_EMIT : t == VK_M_DIELECTRIC ? VKQ_DIEL
                                  : (t == VK_M_LAMBERTIAN || t == VK_M_ISOTROPIC) ? VKQ_DIFF : VKQ_NONE;
                if (mc != (uint32_t)CLS) atomicAdd(&buf.counters[5], 1ull);
#endif
                if constexpr (CLS == VKQ_EMIT) {
                    alive = shade_emitter(sc, rec, rec.m, beta, L);
                } else {
                    const uint4 r = rng.block(depth, 0u); // (BounceXiPhilox::block0)
                    if constexpr (CLS == VKQ_DIEL) alive = shade_dielectric(rec, rec.m, r, o, d);
                    else alive = shade_diffuse(sc, rec, rec.m, rec.m.x, r, o, d, beta, valid);
                }
            }
            if (alive && ++depth > a.max_depth) alive = false; // `depth > MAX_DEPTH` -> 0 (src/main.rs:126)
            if (alive && !(finite3(d) && finite3(o))) {          // the reference's sample is NaN here (see vk_kernels.cu)
                valid = false;
                alive = false;
            }
        }
        if (alive) {
            S.ro[slot] = make_float4(o.x, o.y, o.z, time);
            S.rd[slot] = make_float4(d.x, d.y, d.z, __uint_as_float(depth));
            S.bt[slot] = make_float4(beta.x, beta.y, beta.z, bt.w);
            S.mark_new(slot);
        } else {
            if (valid && finite3(L)) dom_accumulate(dom, buf, pixel, L);
            else ++n_drop;
            ended = true;
        }
    }
}
// One batch of queue q: SPLIT (the trimmed build's flat kernels without media) runs the shading body of the queue's class,
// chosen by one uniform branch per batch; the regeneration and the queue pushes after it are the same for every class.
template <bool LEGACY, bool FLAT, bool SPLIT = false, class W, class D>
VKD void wq_shade_batch(const DScene& sc, const WqCtx<W>& C, const D& dom, const RenderBuffers& buf, uint32_t q, uint32_t n, uint32_t head, uint32_t& n_drop) {
    W& S = C.S;
    const uint32_t lane = C.lane;
    const bool act = lane < n;
    const uint32_t slot = S.ring[q][(head + (act ? lane : 0u)) & W::RMASK];
    bool alive = false, ended = false;
    if (q == VKQ_END) ended = act; // queued regenerations
    else if constexpr (!SPLIT) wq_shade_slot<LEGACY, FLAT, VKQ_NQ>(sc, C, dom, buf, act, slot, alive, ended, n_drop);
    else if (q == VKQ_DIFF || q == VKQ_DIFFI) wq_shade_slot<LEGACY, FLAT, VKQ_DIFF>(sc, C, dom, buf, act, slot, alive, ended, n_drop);
    else if (q == VKQ_EMIT) wq_shade_slot<LEGACY, FLAT, VKQ_EMIT>(sc, C, dom, buf, act, slot, alive, ended, n_drop);
    else wq_shade_slot<LEGACY, FLAT, VKQ_DIEL>(sc, C, dom, buf, act, slot, alive, ended, n_drop); // (no simple scene has Metal)
    // Regenerate in place when enough lanes ended -- the emitter / miss class does, every lane; in the other classes
    // only a few lanes end (a light-sampled direction below the surface has weight 0): those are queued and
    // regenerated together, with full warps.
    const uint32_t m_end = __ballot_sync(0xFFFFFFFFu, ended);
    bool to_end = false;
    if (q == VKQ_END || (uint32_t)__popc(m_end) >= VKQ_REGEN_MIN) alive = wq_regen(C, dom, ended, slot) || alive;
    else to_end = ended;
    // survivors (and regenerated samples) to the extend queue, queued regenerations to theirs: two ballots
    const uint32_t m_ext = __ballot_sync(0xFFFFFFFFu, alive), m_q = __ballot_sync(0xFFFFFFFFu, to_end);
    const uint2 c_ext = S.ct[VKQ_EXT], c_end = S.ct[VKQ_END];
    if (alive) S.ring[VKQ_EXT][(c_ext.y + __popc(m_ext & C.below)) & W::RMASK] = (uint8_t)slot;
    if (to_end) S.ring[VKQ_END][(c_end.y + __popc(m_q & C.below)) & W::RMASK] = (uint8_t)slot;
    __syncwarp();
    if (lane == 0) {
        S.ct[VKQ_EXT] = make_uint2(c_ext.x + (uint32_t)__popc(m_ext), c_ext.y + (uint32_t)__popc(m_ext));
        if (m_q) S.ct[VKQ_END] = make_uint2(c_end.x + (uint32_t)__popc(m_q), c_end.y + (uint32_t)__popc(m_q));
    }
    __syncwarp();
}

// VKQ_SELFCHECK (debug builds only: scripts/build_variants.sh selfcheck:-DVKQ_SELFCHECK=1, tests/test_zz_warpq_selfcheck_gpu.py).
// compute-sanitizer is closed on this pool, so the queue protocol is checked by the kernel itself, before every scheduling
// decision: every queued index is a valid slot, no slot sits in two queues (or twice in one), and the queues together never
// hold more entries than the warp has slots.  Violations are counted in counters[5]; the test asserts the count is zero
// and that the frame equals the normal build's bit for bit.
#ifndef VKQ_SELFCHECK
#define VKQ_SELFCHECK 0
#endif
template <class W>
VKD void wq_selfcheck(const W& S, const RenderBuffers& buf, uint32_t lane, uint32_t in_flight) {
#if VKQ_SELFCHECK
    uint32_t seen[8] = {0, 0, 0, 0, 0, 0, 0, 0}; // 256 slots, one bit each, OR-reduced over the warp per queue entry
    uint32_t bad = 0, total = 0;
    for (uint32_t q = 0; q < W::NQ; ++q) {
        const uint2 c = S.ct[q];
        total += c.x;
        if (c.x > W::N) ++bad;
        for (uint32_t i0 = 0; i0 < c.x; i0 += 32u) {
            const uint32_t i = i0 + lane;
            const bool have = i < c.x;
            const uint32_t slot = have ? S.ring[q][(c.y - c.x + i) & W::RMASK] : 0u;
            if (have && slot >= W::N) ++bad;
            // a slot twice inside this group of 32: two lanes with the same value
            const uint32_t same = __match_any_sync(0xFFFFFFFFu, have ? slot : 0x10000u + lane);
            if (have && __popc(same) != 1) ++bad;
#pragma unroll
            for (uint32_t w = 0; w < 8; ++w) {
                const uint32_t mine = (have && (slot >> 5) == w) ? (1u << (slot & 31u)) : 0u;
                const uint32_t all = __reduce_or_sync(0xFFFFFFFFu, mine);
                if (mine & seen[w]) ++bad; // already queued (an earlier group or an earlier queue)
                seen[w] |= all;
            }
        }
    }
    if (total + in_flight > W::N) ++bad;
    if (bad) atomicAdd(&buf.counters[5], (unsigned long long)bad);
#else
    (void)S, (void)buf, (void)lane, (void)in_flight;
#endif
}

template <class W>
VKD void wq_init(W& S, uint32_t lane) { // every slot starts in the regeneration queue
    if (lane < W::NQ + (W::NQ & 1u)) S.ct[lane] = make_uint2(0u, 0u);
    for (uint32_t i = lane; i < W::N; i += 32u) S.ring[VKQ_END][i] = (uint8_t)i;
    if (lane == 0) {
        S.left = 0u;
        S.exhausted = 0u;
        S.cur_s = 0u;
        S.cur_y = 0u;
        S.cur_x = 0u;
    }
    __syncwarp();
    if (lane == 0) S.ct[VKQ_END] = make_uint2(W::N, W::N);
    __syncwarp();
}
VKD void wq_flush_counters(const RenderBuffers& buf, uint32_t lane, uint32_t n_rays, uint32_t n_drop, uint32_t n_nodes, uint32_t n_prims) {
    unsigned long long w_rays = n_rays, w_drop = n_drop, w_nodes = n_nodes, w_prims = n_prims;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        w_rays += __shfl_xor_sync(0xFFFFFFFFu, w_rays, off);
        w_drop += __shfl_xor_sync(0xFFFFFFFFu, w_drop, off);
        w_nodes += __shfl_xor_sync(0xFFFFFFFFu, w_nodes, off);
        w_prims += __shfl_xor_sync(0xFFFFFFFFu, w_prims, off);
    }
    if (lane == 0) {
        atomicAdd(&buf.counters[3], w_nodes);
        atomicAdd(&buf.counters[4], w_prims);
        atomicAdd(&buf.counters[0], w_rays);
        if (w_drop) atomicAdd(&buf.counters[1], w_drop);
    }
}


#ifndef VKQ_CAP_BPS
#define VKQ_CAP_BPS 0 // (A/B builds only: run at most this many CTAs per SM although more would fit)
#endif
template <class K> static cudaError_t warpq_prepare(K kernel, size_t smem, int* blocks_per_sm) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    // The occupancy calculator assumes the largest shared-memory carveout, the launch does not ask for it by itself
    // (measured: the 6-CTA configurations ran with 4 resident CTAs).  Ask for exactly what the resident CTAs need and no
    // more: whatever the carveout leaves of the SM's 228 KB is L1, and the BVH kernels' node fetches want it.
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, kernel, 32 * VKQ_WARPS, smem);
    if (e != cudaSuccess) return e;
    if (VKQ_CAP_BPS && *blocks_per_sm > VKQ_CAP_BPS) *blocks_per_sm = VKQ_CAP_BPS;
    const size_t need = (size_t)(*blocks_per_sm < 1 ? 1 : *blocks_per_sm) * (smem + 1024);
    int pct = (int)((need * 100 + 233472 - 1) / 233472);
    pct = pct > 100 ? 100 : pct;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    if (e != cudaSuccess) return e;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, kernel, 32 * VKQ_WARPS, smem);
    if (VKQ_CAP_BPS && *blocks_per_sm > VKQ_CAP_BPS) *blocks_per_sm = VKQ_CAP_BPS;
    return e;
}

} // namespace VK_NS
