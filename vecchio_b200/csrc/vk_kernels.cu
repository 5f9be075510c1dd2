// vk_kernels.cu -- kernels of the sample loop.  Compiled twice (see vk_device.cuh): vkfast / vkstrict.
//
//   k_megakernel   persistent path tracer: one lane = one pixel of an 8x4 warp tile, looping over a
//                  chunk of samples with path regeneration; the bounce loop is the iterative form of
//                  ray_color (src/main.rs:123-153, SURVEY App. F).
//   k_intersect    parity hook: world.hit() for a batch of rays.
#include "vk_device.cuh"

namespace VK_NS {

#ifndef VK_BLOCK
#define VK_BLOCK 128
#endif
// Resident CTAs per SM the register allocation must allow.  Measured on B200 (profiles/): the flat
// kernel gains 20 % going from 4 (122 regs) to 8 (64 regs, a few spills) -- it is latency bound on
// dependent ALU chains and indexed constant loads, so more warps win over fewer spills; the BVH
// kernel was flat between 5 and 8 in round 1.  Round 2's body (profiles/r2_sweep_23.log, 4 / 5 / 6 / 7 / 8 CTAs =
// 114 / 96 / 80 / 72 / 64 registers, 0 / 56 / 290 / 416 / 460 B of spill stores): final scene 43.9 / 42.3 / 42.8 / 44.0 / 44.3 ms,
// bowser 5.11 / 4.92 / 5.40 / 5.50 / 5.85 ms, random spheres at 16 spp 1.24 / 1.18 / 1.21 / 1.20 / 1.20 ms -- five it is
// (256-thread CTAs at the same occupancy: no change).
#ifndef VK_MINB_FLAT
#define VK_MINB_FLAT 8
#endif
#ifndef VK_MINB_BVH
#define VK_MINB_BVH 5
#endif

// Work decomposition (deterministic for a seed whatever the grid):
//   item  = one 8x4 pixel tile x one chunk of samples, fetched by a whole warp from a global queue;
//   unit  = one pixel of the tile x one sample.  The 32 lanes of the warp draw units from a
//           warp-local counter (ballot + popc, no memory traffic): a lane whose path has ended takes
//           the next one, so lanes only idle for the last unit of an item.
// A finished sample goes straight into its pixel's integer accumulators (accumulate_sample).
// A batch of frames: item = frame x chunk x tile, frame outermost.  A list of pixels: a "tile" is 32 consecutive list
// entries (the host sets tiles_x to their number, tiles_y to 1), unit u of an item is entry tile * 32 + (u & 31) x sample
// c0 + (u >> 5).  A list across a batch of frames: the same, and each unit resolves its frame (camera, key, plane) from the
// batch-wide entry it takes, since an item's 32 entries may belong to two frames.
template <bool FLAT, bool MEDIA, bool LEGACY, class D>
VKD void megakernel_body(const DScene& sc, const FlatProgram* flat, const DCamera& cam, const RenderArgs& a,
                         const RenderBuffers& buf, const D& dom) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t lanes_below = (1u << lane) - 1u;
    const uint32_t n_tiles = a.tiles_x * a.tiles_y;
    const uint32_t total = n_tiles * a.n_chunks * dom_frames(dom);
    const uint32_t spp_end = a.spp_begin + a.spp_count;
    uint32_t n_rays = 0, n_drop = 0, n_nodes = 0, n_prims = 0; // per lane: far below 2^32 for any frame

#pragma unroll 1
    for (;;) {
        uint32_t item = 0;
        if (lane == 0) item = (uint32_t)atomicAdd(&buf.counters[2], 1ull);
        item = __shfl_sync(0xFFFFFFFFu, item, 0);
        if (item >= total) break;
        uint32_t f = dom_split_frame(dom, item, n_tiles * a.n_chunks); // frame of the item (a list across frames: of the unit)
        uint32_t pbase = dom_plane(dom, f);                            // its first pixel in the accumulators
        const uint32_t chunk = item / n_tiles, tile = item - chunk * n_tiles;
        const uint32_t px0 = (tile % a.tiles_x) * 8u, py0 = (tile / a.tiles_x) * 4u;
        const uint32_t c0 = a.spp_begin + chunk * a.chunk_spp;
        const uint32_t c1 = min(c0 + a.chunk_spp, spp_end);
        const uint32_t n_units = (c1 - c0) * 32u;
        uint32_t next_unit = 0; // warp-uniform

        PathRng rng;
        rng.pixel = 0;
        rng.sample = 0;
        rng.key = make_uint2(a.seed_lo, a.seed_hi);
        dom_frame_key(dom, a, f, rng);
        float3 o = f3(0.0f, 0.0f, 0.0f), d = o, beta = o, L = o;
        float time = 0.0f;
        uint32_t depth = 0, s = 0, s_end = 0, px = 0, py = 0;
        bool alive = false, valid = true, has_unit = false;
#pragma unroll 1
        for (;;) {
            // ---- unit bookkeeping (warp-synchronous: every lane is here with the full mask) ----
            const bool need = !alive && !(has_unit && s < s_end);
            if (need) has_unit = false;
            const uint32_t want = __ballot_sync(0xFFFFFFFFu, need);
            if (need) {
                const uint32_t u = next_unit + __popc(want & lanes_below);
                // (through copies: px, py and rng.pixel passed by reference would change the single-frame kernels' code)
                uint32_t x = px, y = py, pixel;
                if (u < n_units && mk_unit(dom, a, tile, px0, py0, u, x, y, pixel)) {
                    s = c0 + (u >> 5);
                    s_end = s + 1u;
                    rng.pixel = pixel;
                    has_unit = true;
                    if constexpr (dom_frame_per_unit<D>::value) { // (an item's 32 entries may straddle a frame boundary)
                        f = dom_unit_frame(dom, a, rng);
                        pbase = f * dom.fr.n_pix;
                    }
                }
                px = x;
                py = y;
            }
            next_unit += __popc(want);
            const bool work = alive || (has_unit && s < s_end);
            if (__ballot_sync(0xFFFFFFFFu, work || (need && next_unit < n_units)) == 0u) break;
            if (!work) continue;

            // ---- one path segment ---------------------------------------------------------------
            if (!alive) { // regenerate: this lane starts its next sample while others keep bouncing
                rng.sample = s++;
                camera_get_ray(dom_camera(dom, cam, f), rng, px, py, a.width, a.height, o, d, time);
                beta = f3(1.0f, 1.0f, 1.0f);
                L = f3(0.0f, 0.0f, 0.0f);
                depth = 1; // ray_color(ray, .., 1) src/main.rs:190
                valid = true;
                alive = true;
            }
            MediumXi xi;
            xi.table = nullptr;
            xi.rng = rng;
            xi.depth = depth;
            ++n_rays;
            TraceCounters tc = {0u, 0u};
            const TraceHit h = FLAT ? trace_flat<MEDIA>(sc, *flat, o, d, time, 0.001f, CUDART_INF_F, xi, tc)
                                    : trace<MEDIA>(sc, o, d, time, 0.001f, CUDART_INF_F, xi, tc); // src/main.rs:130
            n_nodes += tc.nodes;
            n_prims += tc.prims;
            if (h.prim == VK_REF_NONE) {
                L = L + beta * miss_color(a, d); // src/main.rs:151
                alive = false;
            } else {
                HitRecD rec;
                resolve_hit(sc, h, o, d, time, false, rec);
                alive = LEGACY ? shade_legacy(sc, rec, rng, depth, o, d, time, beta, L, valid)
                               : shade(sc, rec, rng, depth, o, d, time, beta, L, valid);
                if (alive && ++depth > a.max_depth) alive = false; // `depth > MAX_DEPTH` -> 0 (src/main.rs:126)
                // A non-finite ray (refract()'s sqrt of a rounding-negative number, Q7) makes every
                // comparison of the reference false: it walks the WHOLE BVH, "hits" whichever Rect
                // comes last with t = NaN (Q14) and the sample is then NaN and dropped at
                // main.rs:192 (unless that Rect is an emitter).  Drop the sample directly.
                if (alive && !(finite3(d) && finite3(o))) {
                    valid = false;
                    alive = false;
                }
            }
            if (!alive) { // sample finished: NaN/Inf filter of src/main.rs:191-194
                if (valid && finite3(L)) dom_accumulate(dom, buf, pbase + rng.pixel, L);
                else ++n_drop;
            }
        }
    }
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

// ---------------------------------------------------------------------------------------------------
// Dynamic megakernel for BVH scenes.
//
// Measured (profiles/r1_stress_megakernel_full.md, r1_final_scene_megakernel_full.md): when every
// lane traces one whole ray per loop iteration, the warp waits for its longest traversal -- 4.5 of 32
// lanes active on the 10^6-sphere scene (mean 66 node visits per ray, long tail), 9.3 on the final
// scene.  Here the traversal is the resumable state machine of vk_device.cuh and the warp runs it
// under votes (persistent threads with dynamic re-fill, Aila & Laine 2009):
//
//   traverse:  bounded while-while rounds: up to VK_DYN_NODE_STEPS node visits per lane (a lane stops
//              as soon as it holds a primitive), then one primitive test per lane, then a vote;
//   re-fill:   when fewer than VK_DYN_MIN_ACTIVE lanes are still traversing and an idle lane can get
//              work, the warp leaves the loop; idle lanes shade their hit (src/main.rs:131-149),
//              start their next segment, sample or unit, and join the traversal again.
//
// Units (pixel, sample) come from one global queue, one atomic per re-fill and warp; finished samples
// go into the pixel's integer accumulators, so the image is the same as every other variant's.
#ifndef VK_DYN_MIN_ACTIVE
#define VK_DYN_MIN_ACTIVE 16
#endif
#ifndef VK_DYN_NODE_STEPS
#define VK_DYN_NODE_STEPS 4
#endif
// unit = frame x sample x pixel, frame outermost (a list of pixels: sample x list entry; across frames the entry names the frame)
template <bool MEDIA, class D>
VKD void megakernel_dyn_body(const DScene& sc, const DCamera& cam, const RenderArgs& a, const RenderBuffers& buf,
                             unsigned long long* unit_head, const D& dom) {
    const uint32_t lane = threadIdx.x & 31u, lanes_below = (1u << lane) - 1u;
    const uint32_t n_pixels = dom_pixels(dom, a);
    const unsigned long long n_units = (unsigned long long)n_pixels * a.spp_count * dom_frames(dom);
    uint32_t pbase = 0; // first accumulator pixel of this lane's frame
    uint32_t n_rays = 0, n_drop = 0;
    TraceCounters tc = {0u, 0u};

    PathRng rng;
    rng.pixel = 0;
    rng.sample = 0;
    rng.key = make_uint2(a.seed_lo, a.seed_hi);
    float3 zero3 = f3(0.0f, 0.0f, 0.0f), o = zero3, d = zero3, beta = zero3;
    float time = 0.0f;
    uint32_t depth = 0;
    bool exhausted = false, pending = false; // pending: traversal finished, hit not shaded yet
    Trav T;
    T.ref = VKD_DONE;
    T.sp = 0;
    T.enter = false;
    T.cur_inst = 0;
    T.co = T.cd = T.cinv = zero3;
    T.best.t = 0.0f;
    T.best.prim = VK_REF_NONE;
    T.best.inst = 0;
    T.best.face = 0;
#pragma unroll 1
    for (;;) {
        // ---- re-fill: every lane whose traversal has finished ------------------------------------------
        bool need_unit = false, new_ray = false;
        if (T.ref == VKD_DONE && !(exhausted && !pending)) {
            bool alive = false, valid = true;
            float3 L = f3(0.0f, 0.0f, 0.0f);
            if (pending) {
                pending = false;
                if (T.best.prim == VK_REF_NONE) {
                    L = beta * miss_color(a, d); // src/main.rs:151
                } else {
                    HitRecD rec;
                    resolve_hit(sc, T.best, o, d, time, false, rec);
                    alive = shade(sc, rec, rng, depth, o, d, time, beta, L, valid);
                    if (alive && ++depth > a.max_depth) alive = false; // `depth > MAX_DEPTH` -> 0 (src/main.rs:126)
                    if (alive && !(finite3(d) && finite3(o))) {          // the reference's sample is NaN here
                        valid = false;
                        alive = false;
                    }
                }
                if (!alive) { // sample finished: NaN/Inf filter of src/main.rs:191-194
                    if (valid && finite3(L)) dom_accumulate(dom, buf, pbase + rng.pixel, L);
                    else ++n_drop;
                }
            }
            if (alive) new_ray = true;
            else need_unit = !exhausted;
        }
        const uint32_t mu = __ballot_sync(0xFFFFFFFFu, need_unit);
        if (mu) { // one global atomic per warp and re-fill
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(unit_head, (unsigned long long)__popc(mu));
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
            if (need_unit) {
                unsigned long long u = base + __popc(mu & lanes_below);
                if (u < n_units) {
                    uint32_t f = dom_split_frame(dom, u, (unsigned long long)n_pixels * a.spp_count);
                    pbase = f * n_pixels;
                    dom_frame_key(dom, a, f, rng);
                    const uint32_t sb = (uint32_t)(u / n_pixels);
                    rng.pixel = dom_list_pixel(dom, (uint32_t)(u - (unsigned long long)sb * n_pixels)); // i = y*width + x (src/main.rs:182-183)
                    if constexpr (dom_frame_per_unit<D>::value) {
                        f = dom_unit_frame(dom, a, rng);
                        pbase = f * dom.fr.n_pix;
                    }
                    rng.sample = a.spp_begin + sb;
                    camera_get_ray(dom_camera(dom, cam, f), rng, rng.pixel % a.width, rng.pixel / a.width, a.width, a.height, o, d, time);
                    beta = f3(1.0f, 1.0f, 1.0f);
                    depth = 1;
                    new_ray = true;
                } else {
                    exhausted = true;
                }
            }
        }
        if (new_ray) {
            trav_init(T, sc, o, d, CUDART_INF_F); // world.hit(&r, 0.001, inf) src/main.rs:130
            ++n_rays;
        }
        if (__ballot_sync(0xFFFFFFFFu, T.ref != VKD_DONE) == 0u) break; // nothing in flight, nothing left
        // ---- traverse --------------------------------------------------------------------------------------
        MediumXi xi;
        xi.table = nullptr;
#pragma unroll 1
        for (;;) {
            const bool active = T.ref != VKD_DONE;
            const uint32_t m_act = __ballot_sync(0xFFFFFFFFu, active);
            // an idle lane is worth leaving for if it has a hit to shade or can still get a unit
            const uint32_t m_fill = __ballot_sync(0xFFFFFFFFu, !active && (pending || !exhausted));
            if (m_act == 0u || ((uint32_t)__popc(m_act) < VK_DYN_MIN_ACTIVE && m_fill != 0u)) break;
            // a bounded while-while round between two votes: up to VK_DYN_NODE_STEPS node visits (a lane
            // leaves the loop as soon as it holds a primitive), then one primitive test per lane
#pragma unroll 1
            for (int k = 0; k < VK_DYN_NODE_STEPS && trav_at_node(T); ++k) trav_node_step(T, sc, 0.001f, tc);
            if (T.ref != VKD_DONE && !trav_at_node(T)) {
                xi.rng = rng;
                xi.depth = depth;
                trav_prim_step<MEDIA>(T, sc, o, d, time, 0.001f, xi, tc);
            }
            if (active && T.ref == VKD_DONE) pending = true;
        }
    }
    unsigned long long w_rays = n_rays, w_drop = n_drop, w_nodes = tc.nodes, w_prims = tc.prims;
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
// instantiations: {BVH, flat program} x {scene without / with ConstantMedium} x {HEAD integrator, legacy scatter} x work domain
template <bool MEDIA, class D>
__global__ void __launch_bounds__(VK_BLOCK, VK_MINB_BVH) k_megakernel_dyn(const DScene sc, const DCamera cam, const RenderArgs a,
                                                                      const RenderBuffers buf, unsigned long long* unit_head,
                                                                      const __grid_constant__ D dom) {
    megakernel_dyn_body<MEDIA>(sc, cam, a, buf, unit_head, dom);
}
template <bool MEDIA, bool LEGACY, class D>
__global__ void __launch_bounds__(VK_BLOCK, VK_MINB_BVH) k_megakernel(const DScene sc, const DCamera cam, const RenderArgs a,
                                                                  const RenderBuffers buf, const __grid_constant__ D dom) {
    megakernel_body<false, MEDIA, LEGACY>(sc, nullptr, cam, a, buf, dom);
}
template <bool MEDIA, bool LEGACY, class D>
__global__ void __launch_bounds__(VK_BLOCK, VK_MINB_FLAT) k_megakernel_flat(const DScene sc, const __grid_constant__ FlatProgram flat,
                                                                       const DCamera cam, const RenderArgs a, const RenderBuffers buf,
                                                                       const __grid_constant__ D dom) {
    megakernel_body<true, MEDIA, LEGACY>(sc, &flat, cam, a, buf, dom);
}

template <bool FLAT>
VKD void intersect_body(const DScene& sc, const FlatProgram* flat, const vk_ray* __restrict__ rays, size_t n,
                        const float* __restrict__ medium_xi, vk_hit* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const vk_ray r = rays[i];
    const float3 o = f3(r.origin[0], r.origin[1], r.origin[2]);
    const float3 d = f3(r.direction[0], r.direction[1], r.direction[2]);
    MediumXi xi;
    xi.table = medium_xi ? medium_xi + i * VK_MEDIUM_XI_SLOTS : nullptr;
    xi.rng.pixel = (uint32_t)i;
    xi.rng.sample = (uint32_t)(i >> 32);
    xi.rng.key = make_uint2(0x243F6A88u, 0x85A308D3u);
    xi.depth = 1;
    TraceCounters tc = {0u, 0u};
    const TraceHit h = FLAT ? trace_flat<true>(sc, *flat, o, d, r.time, r.tmin, r.tmax, xi, tc) : trace<true>(sc, o, d, r.time, r.tmin, r.tmax, xi, tc);
    vk_hit q;
    q.prim = h.prim;
    q.face = 0;
    q.mat = 0;
    q.front = 0;
    q.t = 0.0f;
    q.p[0] = q.p[1] = q.p[2] = 0.0f;
    q.normal[0] = q.normal[1] = q.normal[2] = 0.0f;
    q.u = q.v = 0.0f;
    q._pad = 0;
    if (h.prim != VK_REF_NONE) {
        HitRecD rec;
        resolve_hit(sc, h, o, d, r.time, true, rec);
        q.face = h.face;
        q.mat = rec.mat;
        q.front = rec.front;
        q.t = rec.t;
        q.p[0] = rec.p.x; q.p[1] = rec.p.y; q.p[2] = rec.p.z;
        q.normal[0] = rec.normal.x; q.normal[1] = rec.normal.y; q.normal[2] = rec.normal.z;
        q.u = rec.u;
        q.v = rec.v;
    }
    out[i] = q;
}
__global__ void __launch_bounds__(VK_BLOCK) k_intersect(const DScene sc, const vk_ray* __restrict__ rays, size_t n,
                                                        const float* __restrict__ medium_xi, vk_hit* __restrict__ out) {
    intersect_body<false>(sc, nullptr, rays, n, medium_xi, out);
}
__global__ void __launch_bounds__(VK_BLOCK) k_intersect_flat(const DScene sc, const __grid_constant__ FlatProgram flat,
                                                             const vk_ray* __restrict__ rays, size_t n,
                                                             const float* __restrict__ medium_xi, vk_hit* __restrict__ out) {
    intersect_body<true>(sc, &flat, rays, n, medium_xi, out);
}

// vk_eval_batch: the shading-side parity hook (include/vecchio_gpu.h).  One record per thread through the same
// device functions the render kernels call.
__global__ void __launch_bounds__(VK_BLOCK) k_eval(const DScene sc, vk_eval* __restrict__ recs, size_t n, uint32_t n_materials,
                                                   uint32_t n_textures) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    vk_eval e = recs[i];
    const float3 p = f3(e.p[0], e.p[1], e.p[2]);
    if (e.op == VK_EVAL_BOUNCE || e.op == VK_EVAL_BOUNCE_LEGACY) {
        if (e.index < n_materials) {
            HitRecD rec;
            rec.p = p;
            rec.normal = f3(e.normal[0], e.normal[1], e.normal[2]);
            rec.t = e.t;
            rec.u = e.u;
            rec.v = e.v;
            rec.front = e.front ? 1u : 0u;
            rec.mat = e.index;
            rec.m = __ldg(&sc.materials[e.index]);
            float3 o = f3(e.ray_o[0], e.ray_o[1], e.ray_o[2]), d = f3(e.ray_d[0], e.ray_d[1], e.ray_d[2]);
            float3 beta = f3(1.0f, 1.0f, 1.0f), L = f3(0.0f, 0.0f, 0.0f);
            float time = e.ray_time;
            bool valid = true;
            const BounceXiTable xi = {make_uint4(e.xi[0], e.xi[1], e.xi[2], e.xi[3]), e.xi[4]};
            const bool alive = e.op == VK_EVAL_BOUNCE ? shade_xi(sc, rec, xi, o, d, time, beta, L, valid)
                                                      : shade_legacy_xi(sc, rec, xi, o, d, time, beta, L, valid);
            e.alive = alive ? 1u : 0u;
            e.valid = valid ? 1u : 0u;
            e.out_o[0] = o.x; e.out_o[1] = o.y; e.out_o[2] = o.z;
            e.out_d[0] = d.x; e.out_d[1] = d.y; e.out_d[2] = d.z;
            e.out_time = time;
            e.beta[0] = beta.x; e.beta[1] = beta.y; e.beta[2] = beta.z;
            e.L[0] = L.x; e.L[1] = L.y; e.L[2] = L.z;
        }
    } else if (e.op == VK_EVAL_TEXTURE) {
        if (e.index < n_textures) {
            const float3 c = tex_value(sc, e.index, e.u, e.v, p);
            e.beta[0] = c.x; e.beta[1] = c.y; e.beta[2] = c.z;
        }
    } else if (e.op == VK_EVAL_LIGHTS_PDF) {
        e.value = lights_pdf_value(sc, p, f3(e.dir[0], e.dir[1], e.dir[2]));
    } else if (e.op == VK_EVAL_LIGHT_RANDOM) {
        if (e.index < sc.n_lights) {
            const float3 v = light_random(sc, __ldg(&sc.lights[e.index]), p, e.xi[0], e.xi[1], e.xi[2]);
            e.out_d[0] = v.x; e.out_d[1] = v.y; e.out_d[2] = v.z;
        }
    }
    recs[i] = e;
}
cudaError_t launch_eval(const DScene& sc, vk_eval* recs, size_t n, uint32_t n_materials, uint32_t n_textures, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    k_eval<<<(unsigned)((n + VK_BLOCK - 1) / VK_BLOCK), VK_BLOCK, 0, st>>>(sc, recs, n, n_materials, n_textures);
    return cudaGetLastError();
}

__global__ void k_philox_kat(const uint32_t* in6, uint32_t* out4) {
    const uint4 r = philox4x32_10(make_uint4(in6[0], in6[1], in6[2], in6[3]), make_uint2(in6[4], in6[5]));
    out4[0] = r.x; out4[1] = r.y; out4[2] = r.z; out4[3] = r.w;
}

// *unit_head must be zero on the stream before the launch
template <class D>
cudaError_t launch_megakernel_dyn(const DScene& sc, const DCamera& cam, const RenderArgs& a, const RenderBuffers& b,
                                  unsigned long long* unit_head, int sm_count, cudaStream_t st, const D& dom) {
    int bps = 0;
    cudaError_t e = sc.has_media ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_megakernel_dyn<true, D>, VK_BLOCK, 0)
                                 : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_megakernel_dyn<false, D>, VK_BLOCK, 0);
    if (e != cudaSuccess) return e;
    const int grid = sm_count * (bps < 1 ? 1 : bps);
    if (sc.has_media) k_megakernel_dyn<true, D><<<grid, VK_BLOCK, 0, st>>>(sc, cam, a, b, unit_head, dom);
    else k_megakernel_dyn<false, D><<<grid, VK_BLOCK, 0, st>>>(sc, cam, a, b, unit_head, dom);
    return cudaGetLastError();
}
#define VK_MEGA_DISPATCH(CALL_BVH, CALL_FLAT)                                                                         \
    if (flat) {                                                                                                        \
        if (media) { if (legacy) { CALL_FLAT(true, true); } else { CALL_FLAT(true, false); } }                         \
        else { if (legacy) { CALL_FLAT(false, true); } else { CALL_FLAT(false, false); } }                             \
    } else {                                                                                                           \
        if (media) { if (legacy) { CALL_BVH(true, true); } else { CALL_BVH(true, false); } }                           \
        else { if (legacy) { CALL_BVH(false, true); } else { CALL_BVH(false, false); } }                               \
    }
// the grid is the single-frame kernels' whatever the domain (megakernel_occupancy: same registers); over a pixel list,
// a.tiles_x * a.tiles_y = groups of 32 list entries
template <class D>
cudaError_t launch_megakernel(const DScene& sc, const FlatProgram* flatp, const DCamera& cam, const RenderArgs& a,
                              const RenderBuffers& b, int grid, bool legacy, cudaStream_t st, const D& dom) {
    const bool flat = flatp && flatp->n, media = sc.has_media;
#define VK_LB(M, G) k_megakernel<M, G, D><<<grid, VK_BLOCK, 0, st>>>(sc, cam, a, b, dom)
#define VK_LF(M, G) k_megakernel_flat<M, G, D><<<grid, VK_BLOCK, 0, st>>>(sc, *flatp, cam, a, b, dom)
    VK_MEGA_DISPATCH(VK_LB, VK_LF)
#undef VK_LB
#undef VK_LF
    return cudaGetLastError();
}
#define VK_INSTANTIATE(D)                                                                                              \
    template cudaError_t launch_megakernel_dyn(const DScene&, const DCamera&, const RenderArgs&, const RenderBuffers&, \
                                               unsigned long long*, int, cudaStream_t, const D&);                      \
    template cudaError_t launch_megakernel(const DScene&, const FlatProgram*, const DCamera&, const RenderArgs&,       \
                                           const RenderBuffers&, int, bool, cudaStream_t, const D&);
VK_INSTANTIATE(OneFrame)
VK_INSTANTIATE(FrameArgs)
VK_INSTANTIATE(ListArgs)
VK_INSTANTIATE(FrameListArgs)
#undef VK_INSTANTIATE
cudaError_t launch_intersect(const DScene& sc, const FlatProgram* flat, const vk_ray* rays, size_t n, const float* medium_xi,
                             vk_hit* out, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    const unsigned grid = (unsigned)((n + VK_BLOCK - 1) / VK_BLOCK);
    if (flat && flat->n) k_intersect_flat<<<grid, VK_BLOCK, 0, st>>>(sc, *flat, rays, n, medium_xi, out);
    else k_intersect<<<grid, VK_BLOCK, 0, st>>>(sc, rays, n, medium_xi, out);
    return cudaGetLastError();
}
cudaError_t megakernel_occupancy(bool flat, bool media, bool legacy, int* blocks_per_sm, int* block_threads) {
    *block_threads = VK_BLOCK;
    cudaError_t e = cudaSuccess;
#define VK_OB(M, G) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, k_megakernel<M, G, OneFrame>, VK_BLOCK, 0)
#define VK_OF(M, G) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, k_megakernel_flat<M, G, OneFrame>, VK_BLOCK, 0)
    VK_MEGA_DISPATCH(VK_OB, VK_OF)
#undef VK_OB
#undef VK_OF
    return e;
}
cudaError_t launch_philox_kat(const uint32_t* ctr_key6, uint32_t* out4, cudaStream_t st) {
    k_philox_kat<<<1, 1, 0, st>>>(ctr_key6, out4);
    return cudaGetLastError();
}

} // namespace VK_NS
