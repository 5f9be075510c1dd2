// vk_stepq.cu -- BVH scenes on warp queues with one queue per TRAVERSAL STEP ("step queues").
//
// vk_warpq.cu's BVH kernel keeps one ray per lane in registers and lets the 32 lanes walk their trees side by side.
// Its ncu reports (profiles/r2_final_scene_warpq_bvh_full.md, r2_stress_warpq_bvh_full.md) say what that costs: 11 of 32
// lanes execute the average instruction -- at any moment the lanes of a warp are spread over node visits, sphere tests,
// box tests, instance entries and stack pops -- and the per-lane stack lives in local memory (0.47 GB of DRAM writes for
// a 16-spp frame).  The lane megakernels (vk_kernels.cu) have the same shape with 7.7 lanes.
//
// Here the traversal itself is cut into steps and every step kind has its own queue, next to the shading queues of
// vk_warpq.cuh.  A ray's traversal state lives in its slot in shared memory: the ray in the frame it is traversed in,
// the closest hit so far, the next reference to process and a short stack (the first VKS_SD entries in shared memory,
// deeper ones -- rare -- in a per-warp strip of global memory).  One iteration of a warp:
//
//   pick the fullest queue -> take 32 slots -> run ONE step kind on them, all lanes in the same code:
//     NODE  (queue VKQ_EXT)   a four-wide node visit (wide_node_test), push the far hits, continue with the nearest
//                             (a fresh ray starts here: root reference with the ENTER flag)
//     SPH / BOX               one leaf test, keep the hit if closer, pop
//     LEAF                    everything else: instance chains (enter an instanced sub-BVH or test the wrapped leaf),
//                             moving spheres, rects, ConstantMedium, the EXIT marker of an instance
//     shading classes         wq_shade_batch, as on the flat scenes
//   -> file every slot under the queue of whatever its traversal needs next (one __match_any_sync), or, when its
//      stack ran empty, under the shading class of its hit.
//
// The closest hit does not depend on the visiting order and the variates are keyed per (pixel, sample, depth), so the
// frame is bit-identical to the other variants' (tests/test_gpu_parity.py).  Reference semantics per step are the lane
// traversal's (vk_device.cuh: trav_node_step / trav_prim_step, src/accel.rs:58-83, src/hittable.rs).
#ifndef VKS_PHILOX_CALL
#define VKS_PHILOX_CALL 0 // (measured: the call costs more than the instruction-cache footprint it saves; final scene 59.3 -> 55.3 ms inlined)
#endif
#define VK_PHILOX_CALL VKS_PHILOX_CALL
#include "vk_warpq.cuh"

namespace VK_NS {

#ifndef VKS_N
#define VKS_N 96 // slots per warp, scenes without instanced sub-BVHs
#endif
#ifndef VKS_N_INST
#define VKS_N_INST 104
#endif
#ifndef VKS_RN
#define VKS_RN 128
#endif
#ifndef VKS_SD
#define VKS_SD 4 // stack entries per slot kept in shared memory (deeper ones: global strip).  Measured: 4 beats 8 -- what the
                 // pools do not take of the SM's 228 KB is L1, and the node fetches live in it (profiles/r2_sweep_6.log, _7.log)
#endif
#ifndef VKS_MINB
#define VKS_MINB 4
#endif
#ifndef VKS_MINB_INST
#define VKS_MINB_INST 4
#endif
#ifndef VKS_NODE_STEPS
#define VKS_NODE_STEPS 6 // node visits per batch: lanes whose next reference is a node again go on (a sphere is tested in
                         // between, VKS_INLINE_SPH), the others wait.  Measured: 1 / 3 / 6 / 12 visits: 11.9 / 8.9 / 8.5 / 8.6 ms
#endif
#ifndef VKS_NODE_STEPS_INST
#define VKS_NODE_STEPS_INST 3 // (final scene: 50.6 ms with 3, 51.4 with 6)
#endif
#ifndef VKS_LEAF_STEPS
#define VKS_LEAF_STEPS 2
#endif
// A queue per leaf kind only pays when each of them can fill a warp.  Scenes with instanced sub-BVHs are the heterogeneous
// ones (final scene: boxes, spheres, moving sphere, media, instance chains, a rect) and their slots are larger, so fewer:
// there every leaf goes through the one generic queue -- its batch runs each kind present at partial lanes, but pays the
// pop / load / store / file overhead once instead of once per kind.
#ifndef VKS_MERGE
#define VKS_MERGE 0
#endif
#ifndef VKS_MERGE_INST
#define VKS_MERGE_INST 1
#endif
#ifndef VKS_INLINE_SPH
#define VKS_INLINE_SPH 1
#endif
#ifndef VKS_PREFETCH
#define VKS_PREFETCH 0 // 1: when a slot is filed, prefetch what its next step will read (the node's line / the sphere) into L1
#endif
#ifndef VKS_STICKY
#define VKS_STICKY 0 // 1: a stage whose queue still holds a full batch runs again (its code is in the L0 instruction cache);
                     // measured slightly slower (final scene 59.3 against 57.7 ms): the fullest queue first keeps the batches fuller
#endif
#define VKS_FRESH 0xFFFFFFFEu // nx of a slot whose ray segment has just been written: no traversal state yet
#define VKS_ENTER VKD_DUP     // on a node reference: the node's own box has not been tested (world root / instance root)

template <int N_, int RN_, int SD_, bool INST_, bool MERGE_>
struct WqStepWarp {
    static constexpr uint32_t N = N_, RMASK = RN_ - 1, NQ = VKQ_NQ_STEP, SD = SD_;
    static constexpr bool INST = INST_;
    static constexpr bool MERGE = MERGE_; // spheres and boxes go through the generic leaf queue (see VKS_MERGE)
    static_assert((RN_ & (RN_ - 1)) == 0 && RN_ >= N_ && RN_ <= 256, "ring capacity: power of two, >= slots, byte indices");
    float4 ro[N_];                 // world ray: origin.xyz, time
    float4 rd[N_];                 // direction.xyz, bits: depth of the segment
    float4 bt[N_];                 // path weight.xyz, bits: global sample index
    uint4 hp[N_];                  // closest hit so far: t bits, primitive, instance index | face << 28 | has-instance << 31;
                                   // .w: reference of the instance whose sub-BVH is being traversed (0: world frame)
    float4 oo[INST_ ? N_ : 1];     // the ray in that instance's frame
    float4 od[INST_ ? N_ : 1];
    uint32_t px[N_];
    uint32_t nx[N_];               // what the traversal processes next (reference, VKD_DONE never stored; VKS_FRESH: new ray)
    uint32_t stk[SD_][N_];         // traversal stack, level-major
    uint8_t sp[N_];                // stack depth
    uint8_t ring[VKQ_NQ_STEP][RN_];
    uint2 ct[VKQ_NQ_STEP + 2];     // per queue: entries, ring write position (padded for 16-byte loads)
    uint32_t cur_s, cur_y, cur_x, left;
    uint32_t exhausted;
    VKD void mark_new(uint32_t slot) { nx[slot] = VKS_FRESH; }
};

// the fullest of the ten queues (entries << 4 | queue; one max chain, made provably uniform by the reduction: see wq_pick)
template <class W>
VKD bool sq_pick(const W& S, uint32_t last_q, uint32_t& q, uint32_t& n_q, uint32_t& tail_q) {
    const uint4 c01 = *reinterpret_cast<const uint4*>(&S.ct[0]), c23 = *reinterpret_cast<const uint4*>(&S.ct[2]);
    const uint4 c45 = *reinterpret_cast<const uint4*>(&S.ct[4]), c67 = *reinterpret_cast<const uint4*>(&S.ct[6]);
    const uint4 c89 = *reinterpret_cast<const uint4*>(&S.ct[8]);
    uint32_t key = c01.x * 16u + VKQ_EXT;
    key = max(key, c67.z * 16u + VKQ_SPH);
    key = max(key, c89.x * 16u + VKQ_BOX);
    key = max(key, c89.z * 16u + VKQ_LEAF);
    key = max(key, c23.x * 16u + VKQ_EMIT);
    key = max(key, c45.z * 16u + VKQ_DIFF);
    key = max(key, c67.x * 16u + VKQ_DIFFI);
    key = max(key, c23.z * 16u + VKQ_DIEL);
    key = max(key, c45.x * 16u + VKQ_METAL);
    key = max(key, c01.z * 16u + VKQ_END);
#if VKS_STICKY
    {   // the stage that ran last goes first while it can fill a warp (the scheduler loop otherwise changes stage almost
        // every iteration, and each change is a walk through code the 6 KB L0 instruction cache has dropped)
        const uint32_t n_last = S.ct[last_q].x;
        if (n_last >= 32u) key = max(key, (n_last + 4096u) * 16u + last_q);
    }
#endif
    key = __reduce_max_sync(0xFFFFFFFFu, key);
    q = key & 15u;
    const uint2 e = S.ct[q];
    n_q = e.x;
    tail_q = e.y;
    return (key >> 4) != 0u;
}

template <bool MEDIA, bool LEGACY, class W, class D>
VKD void stepq_body(const DScene& sc, const DCamera& cam, const RenderArgs& a, const RenderBuffers& buf, unsigned long long* unit_head,
                    uint32_t* gstack, uint32_t glevels, const D& dom) {
    extern __shared__ __align__(16) unsigned char vkq_raw[];
    const uint32_t lane = threadIdx.x & 31u, below = (1u << lane) - 1u;
    W& S = reinterpret_cast<W*>(vkq_raw)[threadIdx.x >> 5];
    const WqCtx<W> C = wq_ctx(dom, cam, a, S, unit_head, lane);
    uint32_t n_rays = 0, n_drop = 0;
    TraceCounters tc = {0u, 0u};
    const uint32_t miss_cls = wq_black_miss(a) ? (uint32_t)VKQ_END : (uint32_t)VKQ_EMIT;
    // this warp's strip of the overflow stack: entry (level - SD, slot)
    uint32_t* const gst = gstack + (size_t)(blockIdx.x * VKQ_WARPS + (threadIdx.x >> 5)) * glevels * W::N;
    const float tmin = 0.001f; // world.hit(&r, 0.001, inf) src/main.rs:130
    wq_init(S, lane);
    uint32_t q = VKQ_END; // the stage that ran last
#pragma unroll 1
    for (;;) {
        wq_selfcheck(S, buf, lane, 0u);
        uint32_t n_q, tail_q, head;
        if (!sq_pick(S, q, q, n_q, tail_q)) break; // every queue empty: all slots have retired
        const uint32_t n = wq_pop(S, q, n_q, tail_q, 32u, lane, head);
        if (q >= VKQ_END && q <= VKQ_DIFFI) {
            wq_shade_batch<LEGACY, false>(sc, C, dom, buf, q, n, head, n_drop);
            continue;
        }
        wq_converge();
        const bool act = lane < n;
        const uint32_t slot = S.ring[q][(head + (act ? lane : 0u)) & W::RMASK];
        // ---- the slot's traversal state ------------------------------------------------------------------------------
        uint32_t ref = S.nx[slot];
        uint32_t sp = S.sp[slot];
        uint4 hp = S.hp[slot];
        float4 O = S.ro[slot], D = S.rd[slot];
        const float time = O.w;
        if (act && ref == VKS_FRESH) {
            hp = make_uint4(__float_as_uint(CUDART_INF_F), VK_REF_NONE, 0u, 0u);
            sp = 0u;
            ref = VKD_TYPE(sc.root) == VK_T_NODE ? (sc.root | VKS_ENTER) : sc.root; // (BVHNode::hit tests its own box first)
            ++n_rays;
        }
        if (W::INST && hp.w != 0u) {
            O = S.oo[slot];
            D = S.od[slot];
        }
        float3 co = f3(O), cd = f3(D);
        float best_t = __uint_as_float(hp.x);
        auto push = [&](uint32_t r) {
            if (sp < W::SD) S.stk[sp][slot] = r;
            else gst[(sp - W::SD) * W::N + slot] = r;
            ++sp;
        };
        auto pop = [&]() -> uint32_t {
            if (sp == 0u) return VKD_DONE;
            --sp;
            return sp < W::SD ? S.stk[sp][slot] : gst[(sp - W::SD) * W::N + slot];
        };
        const uint32_t hi_inst = hp.w ? (0x80000000u | VKD_INDEX(hp.w)) : 0u; // how a hit inside the current frame names its instance

        if (q == VKQ_EXT) {
            // ---- node visits (BVHNode::hit, src/accel.rs:58-83) -------------------------------------------------------
            const float3 cinv = rcp3(cd);
#pragma unroll 1
            for (int k = 0; k < (W::INST ? VKS_NODE_STEPS_INST : VKS_NODE_STEPS); ++k) {
                const bool go = act && ref != VKD_DONE && VKD_TYPE(ref) == VK_T_NODE;
                if (!__any_sync(0xFFFFFFFFu, go)) break;
                if (go) {
                    const uint32_t ni = VKD_INDEX(ref) & ~VKS_ENTER;
                    bool inside = true;
                    if (ref & VKS_ENTER) { // the world root's / an instanced sub-BVH root's own box
                        const float4 n0 = __ldg(&sc.nodes[2 * ni]), n1 = __ldg(&sc.nodes[2 * ni + 1]);
                        float te;
                        inside = aabb_hit(f3(n0), f3(n1), co, cd, cinv, tmin, best_t, te);
                    }
                    if (inside) {
                        ++tc.nodes;
                        uint32_t r0, r1, r2, r3;
                        wide_node_test(sc, ni, co, cd, cinv, tmin, best_t, r0, r1, r2, r3);
                        if (r3 != VK_REF_NONE) push(r3); // nearest first, the others wait on the stack, farthest deepest
                        if (r2 != VK_REF_NONE) push(r2);
                        if (r1 != VK_REF_NONE) push(r1);
                        ref = r0 != VK_REF_NONE ? r0 : pop();
                    } else {
                        ref = pop();
                    }
                }
#if VKS_INLINE_SPH
                // a lane that now holds a sphere tests it here, between two node visits, instead of going through the sphere
                // queue: the test runs at partial lanes, but the lane saves a queue hop and is back for the next visit
                if (!W::MERGE && act && ref != VKD_DONE && VKD_TYPE(ref) == VK_T_SPHERE) {
                    const float4 s = __ldg(&sc.spheres[VKD_INDEX(ref)]);
                    float t;
                    ++tc.prims;
                    if (sphere_t(f3(s), s.w, co, cd, tmin, best_t, t)) {
                        best_t = t;
                        hp.x = __float_as_uint(t);
                        hp.y = ref & ~VKD_DUP;
                        hp.z = hi_inst;
                    }
                    ref = pop();
                }
#endif
            }
        } else if (q == VKQ_SPH) {
            // ---- Sphere::hit (src/hittable.rs:62-102), distance only ------------------------------------------------------
#pragma unroll 1
            for (int k = 0; k < VKS_LEAF_STEPS; ++k) {
                const bool go = act && ref != VKD_DONE && VKD_TYPE(ref) == VK_T_SPHERE;
                if (!__any_sync(0xFFFFFFFFu, go)) break;
                if (go) {
                    const float4 s = __ldg(&sc.spheres[VKD_INDEX(ref)]);
                    float t;
                    ++tc.prims;
                    if (sphere_t(f3(s), s.w, co, cd, tmin, best_t, t)) {
                        best_t = t;
                        hp.x = __float_as_uint(t);
                        hp.y = ref & ~VKD_DUP;
                        hp.z = hi_inst;
                    }
                    ref = pop();
                }
            }
        } else if (q == VKQ_BOX) {
            // ---- Boxy::hit (src/hittable.rs:381-394) ------------------------------------------------------------------------
            const float3 cinv = rcp3(cd);
#pragma unroll 1
            for (int k = 0; k < VKS_LEAF_STEPS; ++k) {
                const bool go = act && ref != VKD_DONE && VKD_TYPE(ref) == VK_T_BOX;
                if (!__any_sync(0xFFFFFFFFu, go)) break;
                if (go) {
                    const uint32_t i = VKD_INDEX(ref);
                    const float4 b0 = __ldg(&sc.boxes[2 * i]), b1 = __ldg(&sc.boxes[2 * i + 1]);
                    float t;
                    uint32_t face = 0;
                    ++tc.prims;
                    if (box_t(f3(b0), f3(b1), co, cd, cinv, tmin, best_t, t, face)) {
                        best_t = t;
                        hp.x = __float_as_uint(t);
                        hp.y = ref & ~VKD_DUP;
                        hp.z = hi_inst | (face << 28);
                    }
                    ref = pop();
                }
            }
        } else {
            // ---- the other leaves (all leaves when W::MERGE): trav_prim_step's cases ------------------------------------
#pragma unroll 1
            for (int k = 0; k < VKS_LEAF_STEPS; ++k) {
                const uint32_t type = VKD_TYPE(ref);
                const bool go = act && ref != VKD_DONE && type != VK_T_NODE && (W::MERGE || (type != VK_T_SPHERE && type != VK_T_BOX));
                if (!__any_sync(0xFFFFFFFFu, go)) break;
                if (go) {
                    bool entered = false;
                    if (type == VKD_T_EXIT) { // leave the instanced sub-BVH: back to the world ray
                        hp.w = 0u;
                        co = f3(S.ro[slot]);
                        cd = f3(S.rd[slot]);
                    } else if (type != VK_T_NONE) {
                        float3 to = co, td = cd;
                        uint32_t leaf = ref, inst = hp.w;
                        if (type == VK_T_XFORM) {
                            leaf = chain_down(sc, ref, to, td) | (ref & VKD_DUP);
                            inst = ref & ~VKD_DUP;
                            if (W::INST && VKD_TYPE(leaf) == VK_T_NODE) { // instanced sub-BVH: traverse it in object space
                                push(VKD_T_EXIT << 28);
                                S.oo[W::INST ? slot : 0u] = make_float4(to.x, to.y, to.z, 0.0f);
                                S.od[W::INST ? slot : 0u] = make_float4(td.x, td.y, td.z, 0.0f);
                                hp.w = inst;
                                ref = (leaf & ~VKD_DUP) | VKS_ENTER;
                                entered = true;
                            }
                        }
                        if (!entered) {
                            float t;
                            uint32_t face = 0;
                            bool hit;
                            ++tc.prims;
                            if (MEDIA && VKD_TYPE(leaf) == VK_T_MEDIUM) {
                                MediumXi xi;
                                xi.table = nullptr;
                                xi.depth = __float_as_uint(S.rd[slot].w);
                                xi.rng.key = make_uint2(a.seed_lo, a.seed_hi);
                                xi.rng.pixel = S.px[slot];
                                xi.rng.sample = __float_as_uint(S.bt[slot].w);
                                dom_slot_rng(dom, a, xi.rng);
                                hit = medium_t(sc, leaf, to, td, time, tmin, best_t, xi, t);
                            } else {
                                hit = leaf_t(sc, leaf, to, td, rcp3(td), time, tmin, best_t, t, face);
                            }
                            if (hit) {
                                best_t = t;
                                hp.x = __float_as_uint(t);
                                hp.y = leaf & ~VKD_DUP;
                                hp.z = (inst ? (0x80000000u | VKD_INDEX(inst)) : 0u) | (face << 28);
                            }
                        }
                    }
                    if (!entered) ref = pop();
                }
            }
        }
        // ---- store the state, file the slot under what it needs next ------------------------------------------------------
        uint32_t cls = VKQ_NONE;
        if (act) {
            S.hp[slot] = hp;
            if (ref == VKD_DONE) {
                if (hp.y == VK_REF_NONE) cls = miss_cls;
                else { // (wq_class_of's answer from the per-primitive table: one byte load for the few lanes that finish)
                    const uint32_t c = __ldg(&sc.prim_cls[sc.cls_base[VKD_TYPE(hp.y)] + VKD_INDEX(hp.y)]);
                    cls = c == 3u ? ((!W::MERGE && (hp.z & 0x80000000u)) ? (uint32_t)VKQ_DIFFI : (uint32_t)VKQ_DIFF) : (uint32_t)VKQ_EMIT + c;
                }
            } else {
                S.nx[slot] = ref;
                S.sp[slot] = (uint8_t)sp;
                const uint32_t type = VKD_TYPE(ref);
#if VKS_PREFETCH
                if (type == VK_T_NODE) asm volatile("prefetch.global.L1 [%0];" ::"l"(sc.wnodes + 8u * (size_t)VKD_INDEX(ref)));
                else if (type == VK_T_SPHERE) asm volatile("prefetch.global.L1 [%0];" ::"l"(sc.spheres + VKD_INDEX(ref)));
#endif
                cls = type == VK_T_NODE ? (uint32_t)VKQ_EXT
                      : (!W::MERGE && type == VK_T_SPHERE) ? (uint32_t)VKQ_SPH
                      : (!W::MERGE && type == VK_T_BOX)    ? (uint32_t)VKQ_BOX
                                                           : (uint32_t)VKQ_LEAF;
            }
        }
        wq_push(S, cls, slot, lane, below);
    }
    wq_flush_counters(buf, lane, n_rays, n_drop, tc.nodes, tc.prims);
}

using WqStepWorld = WqStepWarp<VKS_N, VKS_RN, VKS_SD, false, VKS_MERGE != 0>;
using WqStepInst = WqStepWarp<VKS_N_INST, VKS_RN, VKS_SD, true, VKS_MERGE_INST != 0>;

// instantiations: {no medium, medium} x {HEAD integrator, legacy scatter} x work domain
template <bool MEDIA, bool LEGACY, class D>
__global__ void __launch_bounds__(32 * VKQ_WARPS, VKS_MINB) k_stepq(const DScene sc, const DCamera cam, const RenderArgs a, const RenderBuffers buf,
                                                                unsigned long long* unit_head, uint32_t* gstack, uint32_t glevels,
                                                                const __grid_constant__ D dom) {
    stepq_body<MEDIA, LEGACY, WqStepWorld>(sc, cam, a, buf, unit_head, gstack, glevels, dom);
}
template <bool MEDIA, bool LEGACY, class D>
__global__ void __launch_bounds__(32 * VKQ_WARPS, VKS_MINB_INST) k_stepq_inst(const DScene sc, const DCamera cam, const RenderArgs a, const RenderBuffers buf,
                                                                          unsigned long long* unit_head, uint32_t* gstack, uint32_t glevels,
                                                                          const __grid_constant__ D dom) {
    stepq_body<MEDIA, LEGACY, WqStepInst>(sc, cam, a, buf, unit_head, gstack, glevels, dom);
}

// What the launch needs of the overflow stack: `words` 32-bit words for a scene whose traversal may hold `stack_need`
// entries (vk_scene_info); 0 when the shared-memory part is enough.
size_t stepq_stack_words(uint32_t stack_need, bool inst, int sm_count, uint32_t* levels) {
    *levels = stack_need > VKS_SD ? stack_need - VKS_SD : 0u;
    const size_t warps = (size_t)sm_count * 8 * VKQ_WARPS; // (at most 8 resident CTAs per SM, whatever the occupancy comes to)
    return warps * *levels * (inst ? VKS_N_INST : VKS_N);
}

template <class D>
cudaError_t launch_stepq(const DScene& sc, const DCamera& cam, const RenderArgs& a, const RenderBuffers& b, unsigned long long* unit_head,
                         uint32_t* gstack, uint32_t glevels, bool inst, int sm_count, bool legacy, cudaStream_t st, const D& dom) {
    int bps = 0;
    cudaError_t e;
    const bool media = sc.has_media != 0u;
#define VKS_LAUNCH(KERNEL, WARP)                                                                                       \
    {                                                                                                                  \
        const size_t smem = VKQ_WARPS * sizeof(WARP);                                                                  \
        if ((e = warpq_prepare(KERNEL, smem, &bps)) != cudaSuccess) return e;                                          \
        if (bps > 8) bps = 8;                                                                                          \
        KERNEL<<<sm_count * (bps < 1 ? 1 : bps), 32 * VKQ_WARPS, smem, st>>>(sc, cam, a, b, unit_head, gstack, glevels, dom); \
    }
    if (inst) {
        if (media) { if (legacy) VKS_LAUNCH((k_stepq_inst<true, true, D>), WqStepInst) else VKS_LAUNCH((k_stepq_inst<true, false, D>), WqStepInst) }
        else { if (legacy) VKS_LAUNCH((k_stepq_inst<false, true, D>), WqStepInst) else VKS_LAUNCH((k_stepq_inst<false, false, D>), WqStepInst) }
    } else {
        if (media) { if (legacy) VKS_LAUNCH((k_stepq<true, true, D>), WqStepWorld) else VKS_LAUNCH((k_stepq<true, false, D>), WqStepWorld) }
        else { if (legacy) VKS_LAUNCH((k_stepq<false, true, D>), WqStepWorld) else VKS_LAUNCH((k_stepq<false, false, D>), WqStepWorld) }
    }
#undef VKS_LAUNCH
    return cudaGetLastError();
}
#define VKS_INSTANTIATE(D)                                                                                             \
    template cudaError_t launch_stepq(const DScene&, const DCamera&, const RenderArgs&, const RenderBuffers&, unsigned long long*, \
                                      uint32_t*, uint32_t, bool, int, bool, cudaStream_t, const D&);
VKS_INSTANTIATE(OneFrame)
VKS_INSTANTIATE(FrameArgs)
VKS_INSTANTIATE(ListArgs)
VKS_INSTANTIATE(FrameListArgs)
#undef VKS_INSTANTIATE

} // namespace VK_NS
