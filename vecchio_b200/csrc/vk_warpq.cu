// vk_warpq.cu -- the persistent megakernel as a wavefront inside each WARP ("warp queues").
//
// Round 1's staged kernel (vk_staged.cu) ran generate / extend / sort / shade as CTA-wide stages over a slot
// pool in shared memory.  Its ncu report (profiles/r1_cornell_staged_full.md) names what that costs: 14 % of
// the PC samples sit on the three __syncthreads() of an iteration, the class lists are consumed in order so
// every class border and every list tail is a partial warp (24.9 of 32 lanes), all eight warps of a CTA run
// the same stage at the same time (the ALU-heavy extend of one cannot overlap the MUFU / memory-heavy shade of
// another) and the rotated-box hits shade inside the diffuse class at 5.1 lanes.
//
// Here every warp is its own wavefront machine and nothing is ever synchronised across warps:
//
//   * a warp owns 120 - 176 path slots in shared memory (68 B each) and one ring
//     buffer of slot indices per QUEUE: rays to extend, samples to regenerate, and one queue per shading
//     class (emitter / miss, dielectric, metal, diffuse, diffuse behind an instance chain);
//   * each iteration the warp takes up to 32 entries (extend: 32 x K, K rays per lane through the flat
//     program for instruction-level parallelism) from its FULLEST queue and runs that one stage on them, so
//     the 32 lanes execute one code path; what is left in a queue simply waits for the next entries -- no
//     partial warps at class borders, the pool only has to be large enough that some queue is full;
//   * the results are appended to the queues of the next stage with one __match_any_sync per batch; counters
//     live in shared memory and are touched by this warp alone (no atomics, __syncwarp only);
//   * units (pixel, sample) come from one global counter in chunks of 256 per warp; a finished sample goes
//     into its pixel's integer accumulators (RenderBuffers), so the image does not depend on any of this
//     scheduling and is bit-identical to the other variants for a seed.
//
// Reference semantics are untouched: extend = world.hit (src/main.rs:130) through the same trace functions,
// shade = the same resolve_hit + shade of vk_device.cuh (src/main.rs:131-149), sample end = the NaN filter
// of src/main.rs:191-194, regeneration = Camera::get_ray (src/main.rs:187-190).
#include "vk_warpq.cuh"

namespace VK_NS {

// ---- flat scenes: extend = K rays per lane through the flat program, one queue batch at a time ----------------------
// HYBRID: the program's homogeneous subtrees (FlatProgram::bvh: the final scene's box field and its instanced sphere
// cluster) are traversed inside the extend stage, every lane for its own ray; what differs between the lanes of a batch is
// then only how long a walk through ONE kind of tree takes -- the heterogeneous top of the scene (loose spheres, media,
// rects) is typed batches, and the shading runs on whole batches of a class.
// SHAPE: FlatShape<> walks the program as it comes (trace_flat_k); a compiled shape traces it with trace_flat_static.
// The kernel of a compiled shape also shades each batch with the body of its queue's class (wq_shade_batch's SPLIT): the
// queue number is warp-uniform, so the choice is one uniform branch per batch, and the shading code of a batch has no test
// on the material's type.  (The generic kernel keeps one shading body: with the split it LOST 6 % on Cornell, 32.96
// against 30.96 ms per frame -- a larger kernel around the same rolled trace; with the static trace the two together run
// 26.98 ms, profiles/r3_static_flat_split_b200.jsonl.)
#ifndef VKQ_CLASS_SHADE
#define VKQ_CLASS_SHADE 1
#endif
template <bool MEDIA, bool LEGACY, class W, int K, bool HYBRID, class D, class SHAPE = FlatShape<>>
VKD void warpq_flat_body(const DScene& sc, const FlatProgram* flat, const DCamera& cam, const RenderArgs& a, const RenderBuffers& buf,
                         unsigned long long* unit_head, const D& dom) {
    extern __shared__ __align__(16) unsigned char vkq_raw[];
    const uint32_t lane = threadIdx.x & 31u, below = (1u << lane) - 1u;
    W& S = reinterpret_cast<W*>(vkq_raw)[threadIdx.x >> 5];
    const WqCtx<W> C = wq_ctx(dom, cam, a, S, unit_head, lane);
    uint32_t n_rays = 0, n_drop = 0, n_prims = 0;
    TraceCounters tc = {0u, 0u};
    constexpr uint32_t EXT_CAP = 32u * K;
    // a miss under the constant black background of src/main.rs:124 adds nothing: the slot goes straight to regeneration
    const uint32_t miss_cls = wq_black_miss(a) ? (uint32_t)VKQ_END : (uint32_t)VKQ_EMIT;
    wq_init(S, lane);
#pragma unroll 1
    for (;;) {
        uint32_t q, n_q, tail_q, head;
        wq_selfcheck(S, buf, lane, 0u);
        if (!wq_pick(S, wq_counts(S), EXT_CAP, q, n_q, tail_q)) break; // every queue is empty: all slots have retired
        const uint32_t n = wq_pop(S, q, n_q, tail_q, q == VKQ_EXT ? EXT_CAP : 32u, lane, head);
        if (q != VKQ_EXT) {
            constexpr bool SPLIT = VKQ_CLASS_SHADE && SHAPE::n_segs != 0;
            wq_shade_batch<LEGACY, !HYBRID, SPLIT>(sc, C, dom, buf, q, n, head, n_drop); // (no shading records for subtree hits)
            continue;
        }
        // ---- extend: world.hit() (src/main.rs:130) for up to EXT_CAP rays, K per lane --------------------------------
        wq_converge();
        float3 o[K], d[K];
        float tm[K], best_t[K];
        bool live[K];
        uint32_t best_hit[K], slot[K];
        MediumXi xi[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const uint32_t e = lane + 32u * k;
            live[k] = e < n;
            slot[k] = S.ring[VKQ_EXT][(head + (live[k] ? e : 0u)) & W::RMASK];
            const float4 ro = S.ro[slot[k]], rd = S.rd[slot[k]];
            o[k] = f3(ro);
            d[k] = f3(rd);
            tm[k] = ro.w;
            xi[k].table = nullptr;
            xi[k].depth = __float_as_uint(rd.w);
            xi[k].rng.key = make_uint2(a.seed_lo, a.seed_hi);
            xi[k].rng.pixel = MEDIA ? S.px[slot[k]] : 0u;
            xi[k].rng.sample = MEDIA ? __float_as_uint(S.bt[slot[k]].w) : 0u;
            if (MEDIA) dom_slot_rng(dom, a, xi[k].rng);
        }
        TraceHit sub[K];
#if !VK_STRICT
        if constexpr (SHAPE::n_segs != 0) {
            static_assert(!MEDIA && !HYBRID, "a compiled shape has no media and no subtrees");
            trace_flat_static<K>(*flat, SHAPE{}, o, d, 0.001f, best_t, best_hit);
        } else
#endif
            trace_flat_k<K, MEDIA, HYBRID>(sc, *flat, o, d, tm, live, 0.001f, xi, best_t, best_hit, sub, &tc);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            uint32_t cls = VKQ_NONE;
            if (live[k]) {
                ++n_rays;
                n_prims += flat->n;
                uint32_t prim = VK_REF_NONE, hi = 0u;
                cls = miss_cls; // a miss ends the sample like an emitter does
                if (HYBRID && best_hit[k] == 0xFFFFFFFEu) { // the closest hit came from a subtree
                    prim = sub[k].prim;
                    hi = (sub[k].inst ? (0x80000000u | VKD_INDEX(sub[k].inst)) : 0u) | (sub[k].face << 28);
                    cls = wq_class_of(sc, prim, sub[k].inst);
                } else if (best_hit[k] != 0xFFFFFFFFu) {
                    // the trace returns class-tagged ids: the ray is filed without a look at its entry; the shade stage finds
                    // the leaf and its instance under the entry (DScene::flat_shade) if it needs them at all
                    cls = best_hit[k] >> 8;
                    best_hit[k] = VKF_HIT_INDEX(best_hit[k]);
                    prim = 1u; // (anything but VK_REF_NONE)
                    if (HYBRID) { // (no shading records for a hybrid program: the slot carries the leaf itself)
                        const FlatHit& fh = flat->hits[best_hit[k]];
                        prim = fh.prim & ~VKD_DUP;
                        hi = (fh.inst ? (0x80000000u | VKD_INDEX(fh.inst)) : 0u) | (fh.face << 28);
                    }
                }
                S.hp[slot[k]] = make_uint4(__float_as_uint(best_t[k]), prim, hi, best_hit[k]); // .w: entry of the flat program's hit table
            }
            if (k == 0 || n > 32u * k) wq_push(S, cls, slot[k], lane, below); // (warp-uniform condition)
        }
    }
    wq_flush_counters(buf, lane, n_rays, n_drop, tc.nodes, n_prims + tc.prims);
}

// ---- BVH scenes: extend = the resumable traversal (Trav, vk_device.cuh) with dynamic fetch ------------------------------
// Traversal lengths differ by orders of magnitude between rays (10^6 spheres: mean 28 four-wide visits, some hundreds),
// so a lane is not tied to a batch: every lane keeps ONE ray's traversal in registers (stack in local memory) and the
// warp steps all of them in bounded while-while rounds.  A round costs one vote beyond the traversal itself; only when
// VKQ_BVH_IDLE lanes have nothing left to traverse does the warp do a TURNOVER: the finished rays store their hits and
// are filed under their shading classes, the idle lanes take the next entries of the extend queue, and if that queue
// could not feed them the warp shades one full batch of the fullest class -- its other rays stay in flight in
// registers -- which refills the extend queue.  Shading therefore always runs on whole batches of one class, and
// traversal with at most VKQ_BVH_IDLE - 1 idle lanes.  (First version: fetch and retire in every round, whenever one
// lane was idle or finished -- ~190 instructions of bookkeeping per ~300 of traversal, half the lane megakernel's speed.)
#ifndef VKQ_BVH_IDLE
#define VKQ_BVH_IDLE 8u
#endif
#ifndef VKQ_NODE_STEPS
#define VKQ_NODE_STEPS 4
#endif
template <bool MEDIA, bool LEGACY, class W, class D>
VKD void warpq_bvh_body(const DScene& sc, const DCamera& cam, const RenderArgs& a, const RenderBuffers& buf, unsigned long long* unit_head,
                        const D& dom) {
    extern __shared__ __align__(16) unsigned char vkq_raw[];
    const uint32_t lane = threadIdx.x & 31u, below = (1u << lane) - 1u;
    W& S = reinterpret_cast<W*>(vkq_raw)[threadIdx.x >> 5];
    const WqCtx<W> C = wq_ctx(dom, cam, a, S, unit_head, lane);
    uint32_t n_rays = 0, n_drop = 0;
    TraceCounters tc = {0u, 0u};
    const uint32_t miss_cls = wq_black_miss(a) ? (uint32_t)VKQ_END : (uint32_t)VKQ_EMIT;
    wq_init(S, lane);

    Trav T; // this lane's ray in flight (T.ref == VKD_DONE: none)
    T.ref = VKD_DONE;
    T.sp = 0;
    T.enter = false;
    T.cur_inst = 0;
    T.co = T.cd = T.cinv = f3(0.0f, 0.0f, 0.0f);
    T.best.t = 0.0f;
    T.best.prim = VK_REF_NONE;
    T.best.inst = 0;
    T.best.face = 0;
    float3 o = f3(0.0f, 0.0f, 0.0f), d = o;
    float tm = 0.0f;
    uint32_t cur = 0xFFFFFFFFu; // slot of the ray in flight
    MediumXi xi;
    xi.table = nullptr;
    xi.depth = 0;
    xi.rng.key = make_uint2(a.seed_lo, a.seed_hi);
    xi.rng.pixel = 0;
    xi.rng.sample = 0;
#pragma unroll 1
    for (;;) {
        // ---- turnover, only when VKQ_BVH_IDLE lanes have nothing to traverse (one vote per round otherwise): retire the
        // finished rays, fetch new ones for every idle lane, and if the extend queue could not feed them, shade a batch
        const bool done_lane = T.ref == VKD_DONE;
        const uint32_t m_done = __ballot_sync(0xFFFFFFFFu, done_lane);
        if ((uint32_t)__popc(m_done) >= VKQ_BVH_IDLE) {
            const bool fin = done_lane && cur != 0xFFFFFFFFu;
            if (__ballot_sync(0xFFFFFFFFu, fin) != 0u) { // finished rays: the hit, filed under its shading class
                uint32_t cls = VKQ_NONE, slot = 0u;
                if (fin) {
                    slot = cur;
                    cur = 0xFFFFFFFFu;
                    S.hp[slot] = make_uint4(__float_as_uint(T.best.t), T.best.prim,
                                            (T.best.inst ? (0x80000000u | VKD_INDEX(T.best.inst)) : 0u) | (T.best.face << 28), 0u);
                    cls = T.best.prim == VK_REF_NONE ? miss_cls : wq_class_of(sc, T.best.prim, T.best.inst);
                }
                wq_push(S, cls, slot, lane, below);
            }
            wq_selfcheck(S, buf, lane, (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, cur != 0xFFFFFFFFu)));
            const WqCounts cnt = wq_counts(S);
            const uint32_t n_ext = __reduce_max_sync(0xFFFFFFFFu, cnt.c01.x); // (provably uniform, see wq_pick)
            if (n_ext != 0u) { // fetch: the idle lanes take the next rays of the extend queue
                uint32_t head;
                const uint32_t take = wq_pop(S, VKQ_EXT, n_ext, cnt.c01.y, (uint32_t)__popc(m_done), lane, head);
                const uint32_t rank = (uint32_t)__popc(m_done & below);
                if (done_lane && rank < take) {
                    cur = S.ring[VKQ_EXT][(head + rank) & W::RMASK];
                    const float4 ro = S.ro[cur], rd = S.rd[cur];
                    o = f3(ro);
                    d = f3(rd);
                    tm = ro.w;
                    xi.depth = __float_as_uint(rd.w);
                    if (MEDIA) {
                        xi.rng.pixel = S.px[cur];
                        xi.rng.sample = __float_as_uint(S.bt[cur].w);
                        dom_slot_rng(dom, a, xi.rng);
                    }
                    trav_init(T, sc, o, d, CUDART_INF_F); // world.hit(&r, 0.001, inf) src/main.rs:130
                    ++n_rays;
                }
            }
            const uint32_t m_act = __ballot_sync(0xFFFFFFFFu, T.ref != VKD_DONE);
            if (32u - (uint32_t)__popc(m_act) >= VKQ_BVH_IDLE) { // still starved: refill the extend queue from the fullest class
                uint32_t q, n_q, tail_q, head;
                if (wq_pick(S, wq_counts(S), 0u, q, n_q, tail_q)) {
                    const uint32_t n = wq_pop(S, q, n_q, tail_q, 32u, lane, head);
                    wq_shade_batch<LEGACY, false>(sc, C, dom, buf, q, n, head, n_drop);
                    continue;
                }
                if (m_act == 0u) break; // nothing in flight, nothing queued: all slots have retired
            }
        }
        // ---- traverse: a bounded while-while round for every ray in flight ---------------------------------------------
        wq_converge();
#pragma unroll 1
        for (int k = 0; k < VKQ_NODE_STEPS && trav_at_node(T); ++k) trav_node_step(T, sc, 0.001f, tc);
        if (T.ref != VKD_DONE && !trav_at_node(T)) trav_prim_step<MEDIA>(T, sc, o, d, tm, 0.001f, xi, tc);
    }
    wq_flush_counters(buf, lane, n_rays, n_drop, tc.nodes, tc.prims);
}

using WqFlat = WqWarp<VKQ_N_FLAT, VKQ_RN_FLAT>;
using WqMedia = WqWarp<VKQ_N_MEDIA, VKQ_RN_MEDIA>;
using WqBvh = WqWarp<VKQ_N_BVH, VKQ_RN_BVH>;
using WqHyb = WqWarp<VKQ_N_HYB, VKQ_RN_HYB>;
static_assert(VKQ_WARPS <= 15, "one named barrier per warp of the CTA");

// instantiations: {no medium, medium} x {HEAD integrator, legacy scatter} x work domain
template <bool MEDIA, bool LEGACY, class D>
__global__ void __launch_bounds__(32 * VKQ_WARPS, VKQ_MINB_BVH) k_warpq(const DScene sc, const DCamera cam, const RenderArgs a, const RenderBuffers buf,
                                                                    unsigned long long* unit_head, const __grid_constant__ D dom) {
    warpq_bvh_body<MEDIA, LEGACY, WqBvh>(sc, cam, a, buf, unit_head, dom);
}
template <bool LEGACY, class D>
__global__ void __launch_bounds__(32 * VKQ_WARPS, VKQ_MINB_FLAT) k_warpq_flat(const DScene sc, const __grid_constant__ FlatProgram flat, const DCamera cam,
                                                                          const RenderArgs a, const RenderBuffers buf, unsigned long long* unit_head,
                                                                          const __grid_constant__ D dom) {
    warpq_flat_body<false, LEGACY, WqFlat, VKQ_K_FLAT, false>(sc, &flat, cam, a, buf, unit_head, dom);
}
#if VK_SIMPLE
// k_warpq_flat for a program of a compiled shape (FlatShape, vk_internal.h; chosen at upload)
template <class SHAPE, class D>
__global__ void __launch_bounds__(32 * VKQ_WARPS, VKQ_MINB_FLAT) k_warpq_flat_static(const DScene sc, const __grid_constant__ FlatProgram flat,
                                                                                 const DCamera cam, const RenderArgs a, const RenderBuffers buf,
                                                                                 unsigned long long* unit_head, const __grid_constant__ D dom) {
    warpq_flat_body<false, false, WqFlat, VKQ_K_FLAT, false, D, SHAPE>(sc, &flat, cam, a, buf, unit_head, dom);
}
#endif
template <bool LEGACY, class D>
__global__ void __launch_bounds__(32 * VKQ_WARPS, VKQ_MINB_MEDIA) k_warpq_flat_media(const DScene sc, const __grid_constant__ FlatProgram flat,
                                                                                 const DCamera cam, const RenderArgs a, const RenderBuffers buf,
                                                                                 unsigned long long* unit_head, const __grid_constant__ D dom) {
    warpq_flat_body<true, LEGACY, WqMedia, VKQ_K_MEDIA, false>(sc, &flat, cam, a, buf, unit_head, dom);
}
#if !VK_SIMPLE
template <bool MEDIA, bool LEGACY, class D>
__global__ void __launch_bounds__(32 * VKQ_WARPS, VKQ_MINB_HYB) k_warpq_hybrid(const DScene sc, const __grid_constant__ FlatProgram flat, const DCamera cam,
                                                                            const RenderArgs a, const RenderBuffers buf, unsigned long long* unit_head,
                                                                            const __grid_constant__ D dom) {
    warpq_flat_body<MEDIA, LEGACY, WqHyb, 1, true>(sc, &flat, cam, a, buf, unit_head, dom);
}
#endif

// grid = sm_count * resident CTAs (persistent); *unit_head must be zero on the stream before the launch
// flat_shape: the program's compiled shape (VKF_SHAPE_*, found at upload), or VKF_SHAPE_NONE
template <class D>
cudaError_t launch_warpq(const DScene& sc, const FlatProgram* flat, uint32_t flat_shape, const DCamera& cam, const RenderArgs& a,
                         const RenderBuffers& b, unsigned long long* unit_head, int sm_count, bool legacy, cudaStream_t st, const D& dom) {
    int bps = 0;
    cudaError_t e;
    const bool media = sc.has_media != 0u;
#define VKQ_LAUNCH_FLAT(KERNEL, WARP)                                                                                  \
    {                                                                                                                  \
        const size_t smem = VKQ_WARPS * sizeof(WARP);                                                                  \
        if ((e = warpq_prepare(KERNEL, smem, &bps)) != cudaSuccess) return e;                                          \
        KERNEL<<<sm_count * (bps < 1 ? 1 : bps), 32 * VKQ_WARPS, smem, st>>>(sc, *flat, cam, a, b, unit_head, dom);    \
    }
#define VKQ_LAUNCH_BVH(KERNEL)                                                                                         \
    {                                                                                                                  \
        const size_t smem = VKQ_WARPS * sizeof(WqBvh);                                                                 \
        if ((e = warpq_prepare(KERNEL, smem, &bps)) != cudaSuccess) return e;                                          \
        KERNEL<<<sm_count * (bps < 1 ? 1 : bps), 32 * VKQ_WARPS, smem, st>>>(sc, cam, a, b, unit_head, dom);           \
    }
#if VK_SIMPLE
    (void)legacy; // the trimmed build exists for the HEAD integrator on flat scenes only
    if (media) VKQ_LAUNCH_FLAT((k_warpq_flat_media<false, D>), WqMedia)
    else if (flat_shape == VKF_SHAPE_CORNELL) VKQ_LAUNCH_FLAT((k_warpq_flat_static<FlatShapeCornell, D>), WqFlat)
    else VKQ_LAUNCH_FLAT((k_warpq_flat<false, D>), WqFlat)
#else
    (void)flat_shape; // (shapes are compiled into the trimmed build only)
#define VKQ_LAUNCH_HYB(M, G) VKQ_LAUNCH_FLAT((k_warpq_hybrid<M, G, D>), WqHyb)
    if (flat && flat->n && flat->n_bvh) {
        if (media) { if (legacy) VKQ_LAUNCH_HYB(true, true) else VKQ_LAUNCH_HYB(true, false) }
        else { if (legacy) VKQ_LAUNCH_HYB(false, true) else VKQ_LAUNCH_HYB(false, false) }
    } else if (flat && flat->n) {
        if (media) { if (legacy) VKQ_LAUNCH_FLAT((k_warpq_flat_media<true, D>), WqMedia) else VKQ_LAUNCH_FLAT((k_warpq_flat_media<false, D>), WqMedia) }
        else { if (legacy) VKQ_LAUNCH_FLAT((k_warpq_flat<true, D>), WqFlat) else VKQ_LAUNCH_FLAT((k_warpq_flat<false, D>), WqFlat) }
    } else {
        if (media) { if (legacy) VKQ_LAUNCH_BVH((k_warpq<true, true, D>)) else VKQ_LAUNCH_BVH((k_warpq<true, false, D>)) }
        else { if (legacy) VKQ_LAUNCH_BVH((k_warpq<false, true, D>)) else VKQ_LAUNCH_BVH((k_warpq<false, false, D>)) }
    }
#undef VKQ_LAUNCH_HYB
#endif
#undef VKQ_LAUNCH_FLAT
#undef VKQ_LAUNCH_BVH
    return cudaGetLastError();
}
#define VKQ_INSTANTIATE(D)                                                                                             \
    template cudaError_t launch_warpq(const DScene&, const FlatProgram*, uint32_t, const DCamera&, const RenderArgs&,         \
                                      const RenderBuffers&, unsigned long long*, int, bool, cudaStream_t, const D&);
VKQ_INSTANTIATE(OneFrame)
VKQ_INSTANTIATE(FrameArgs)
VKQ_INSTANTIATE(ListArgs)
VKQ_INSTANTIATE(FrameListArgs)
#undef VKQ_INSTANTIATE

} // namespace VK_NS
