// vk_device.cuh -- device functions of the path-tracing sample loop (sm_100a).
//
// Included by vk_kernels.cu, which is compiled twice:
//   VK_STRICT=0 (namespace vkfast)   FMA contraction on, reciprocal slab test, fast intrinsics where
//                                    only the distribution matters.  The render path.
//   VK_STRICT=1 (namespace vkstrict) -fmad=false, IEEE division and sqrt, and the SAME operation
//                                    order as the reference's Rust, so that hit distances are
//                                    bit-identical to the CPU restatement (hit-parity path).
// Every function names the reference code it implements (paths relative to the reference root).
#pragma once
#include <math_constants.h>

#include "vk_internal.h"

#ifndef VK_STRICT
#define VK_STRICT 0
#endif
// VK_SIMPLE=1 (namespace vkfast_simple, vk_staged.cu only): the same code with everything a "simple" scene
// cannot reach compiled out -- non-solid textures, Metal, SpecDiffuse, sphere / box lights, more than
// one light, moving spheres, (u, v).  vk_scene_upload decides whether a scene is simple (Cornell box,
// Cornell smoke).  No arithmetic changes; the point is the instruction footprint: the staged kernel
// stalls on instruction fetch when its hot code does not fit the 32 KB instruction cache.
#ifndef VK_SIMPLE
#define VK_SIMPLE 0
#endif
// VK_LIGHT0=1 (namespace vkfast_l0; vk_kernels.cu, vk_warpq.cu, vk_stepq.cu): the general render build with the light
// list compiled as what every shipped scene has -- exactly one unflipped Rect -- read from the kernel parameters
// (DScene::light0_a / _b) instead of the general list code (Sphere / Boxy lights, several lights, the records behind
// lights[] -> rects[]), and without SpecDiffuse (its choice draws a Philox block of its own, inlined into every shade).
// vk_scene_upload decides (vk_ctx::one_rect_light && !has_specdiffuse); anything else runs namespace vkfast.  A
// REPLACEMENT, so the body shrinks: 4 % on the final scene, bowser, balls and random-spheres scenes; as an extra branch
// next to the general code it LOST 7 % (profiles/r2_sweep_18.log, r2_sweep_22.log).
#ifndef VK_LIGHT0
#define VK_LIGHT0 0
#endif
#if VK_STRICT
#define VK_NS vkstrict
#elif VK_SIMPLE
#define VK_NS vkfast_simple
#elif VK_LIGHT0
#define VK_NS vkfast_l0
#else
#define VK_NS vkfast
#endif

namespace VK_NS {

#define VKD __device__ __forceinline__
#define VK_PI 3.14159265358979323846f

// ---------------------------------------------------------------------------------------------
// Vec3 (src/vec3.rs)
// ---------------------------------------------------------------------------------------------
VKD float3 f3(float x, float y, float z) { return make_float3(x, y, z); }
VKD float3 f3(float4 v) { return make_float3(v.x, v.y, v.z); }
VKD float3 operator+(float3 a, float3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
VKD float3 operator-(float3 a, float3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
VKD float3 operator*(float3 a, float3 b) { return f3(a.x * b.x, a.y * b.y, a.z * b.z); }
VKD float3 operator*(float3 a, float s) { return f3(a.x * s, a.y * s, a.z * s); }
VKD float3 operator/(float3 a, float s) { return f3(a.x / s, a.y / s, a.z / s); }
VKD float3 operator-(float3 a) { return f3(-a.x, -a.y, -a.z); }
VKD float dot3(float3 a, float3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
VKD float3 cross3(float3 a, float3 b) { return f3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
VKD float length2(float3 a) { return a.x * a.x + a.y * a.y + a.z * a.z; }
VKD float3 unit_vector(float3 a) { // src/vec3.rs:39-42 (three divisions by sqrt, no rsqrt)
#if VK_STRICT
    float n = sqrtf(length2(a));
    return f3(a.x / n, a.y / n, a.z / n);
#else
    return a * rsqrtf(length2(a));
#endif
}
VKD float comp(float3 v, uint32_t a) { return a == 0 ? v.x : (a == 1 ? v.y : v.z); }
VKD bool finite3(float3 v) { return isfinite(v.x) && isfinite(v.y) && isfinite(v.z); }
VKD float3 at(float3 o, float3 d, float t) { // Ray::at src/main.rs:51-53 (never contracted: see sphere_t)
    return f3(__fadd_rn(o.x, __fmul_rn(d.x, t)), __fadd_rn(o.y, __fmul_rn(d.y, t)), __fadd_rn(o.z, __fmul_rn(d.z, t)));
}

// ---------------------------------------------------------------------------------------------
// RNG: counter-based Philox4x32-10 (Salmon et al. 2011), key = render seed, counter =
// (pixel, global sample, depth << 8 | block, 0).  Replaces rand::thread_rng() at every call site
// of the hot path (SURVEY App. D); only the distributions are kept.
// ---------------------------------------------------------------------------------------------
// (VK_PHILOX_CALL: one out-of-line copy instead of ~9 inlined ones of 60 instructions each -- the step-queue kernel's
// executed code must stay inside the 32 KB instruction cache, see vk_stepq.cu)
#if defined(VK_PHILOX_CALL) && VK_PHILOX_CALL
static __device__ __noinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#else
VKD uint4 philox4x32_10(uint4 c, uint2 k) {
#endif
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        // the two products as 64-bit multiplies: ptxas then emits ONE IMAD.WIDE.U32 per product; written as __umulhi + a 32-bit
        // multiply it split two products in five into IMAD.HI + IMAD (75 -> 57 multiply instructions in the Cornell kernel; Cornell
        // 31.10 -> 30.96 ms, smoke 18.39 -> 18.23 ms, 10^6 spheres 22.60 -> 22.38 ms, final scene 42.43 -> 42.17 ms, profiles/r2_sweep_25.log)
        const uint64_t p0 = (uint64_t)0xD2511F53u * c.x, p1 = (uint64_t)0xCD9E8D57u * c.z;
        const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}
#if VK_STRICT
VKD float u01(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-8f; } // gen::<f32>(): 24-bit [0,1)
#else
// 23-bit grid built with integer ops only (I2F runs on the quarter-rate XU pipe); the reference's
// 24-bit grid and this one are indistinguishable at any spp a render uses
VKD float u01(uint32_t x) { return __uint_as_float(0x3F800000u | (x >> 9)) - 1.0f; }
#endif
VKD float gen_range(uint32_t x, float lo, float hi) {                           // gen_range(lo,hi): 23-bit [lo,hi)
    const float scale = hi - lo;
    const float res = __uint_as_float(0x3F800000u | (x >> 9)) * scale + (lo - scale);
    return res < hi ? res : lo; // rand 0.7.3 redraws on the 2^-24 rounding event
}
struct PathRng {
    uint32_t pixel, sample;
    uint2 key;
    VKD uint4 block(uint32_t depth, uint32_t blk, uint32_t w = 0u) const {
        return philox4x32_10(make_uint4(pixel, sample, (depth << 8) | blk, w), key);
    }
};
// Source of the ConstantMedium free-flight variate (src/hittable.rs:473): an injected table for
// vk_intersect (VK_MEDIUM_XI_SLOTS entries per ray: scenes of up to four media), and for the render
// Philox block 1 of the current segment with the counter's fourth word counting groups of four
// (medium, visit) pairs -- every medium of a scene draws independently, however many there are.
struct MediumXi {
    const float* table; // VK_MEDIUM_XI_SLOTS per ray, or nullptr
    PathRng rng;
    uint32_t depth;
    VKD float get(uint32_t medium_index, uint32_t second_visit) const {
        const uint32_t slot = medium_index * 2u + second_visit;
        if (table) return table[slot % VK_MEDIUM_XI_SLOTS];
        const uint4 b = rng.block(depth, 1u, slot >> 2);
        const uint32_t w = (slot & 3u) == 0 ? b.x : ((slot & 3u) == 1 ? b.y : ((slot & 3u) == 2 ? b.z : b.w));
        return u01(w);
    }
};

// ---------------------------------------------------------------------------------------------
// AxisBB::hit (src/accel.rs:16-35).  f32::min/max and fminf/fmaxf both return the non-NaN operand.
// The reference's per-axis early exit is equivalent to one test after the third axis (the
// interval only shrinks).  STRICT divides like the reference; FAST multiplies by 1/d.
// ---------------------------------------------------------------------------------------------
VKD bool aabb_hit(float3 bmin, float3 bmax, float3 o, float3 d, float3 inv_d, float tmin, float tmax, float& t_entry) {
#if VK_STRICT
    (void)inv_d;
    const float ax = (bmin.x - o.x) / d.x, bx = (bmax.x - o.x) / d.x;
    const float ay = (bmin.y - o.y) / d.y, by = (bmax.y - o.y) / d.y;
    const float az = (bmin.z - o.z) / d.z, bz = (bmax.z - o.z) / d.z;
#else
    (void)d;
    const float ax = (bmin.x - o.x) * inv_d.x, bx = (bmax.x - o.x) * inv_d.x;
    const float ay = (bmin.y - o.y) * inv_d.y, by = (bmax.y - o.y) * inv_d.y;
    const float az = (bmin.z - o.z) * inv_d.z, bz = (bmax.z - o.z) * inv_d.z;
#endif
    tmin = fmaxf(fminf(ax, bx), tmin);
    tmax = fminf(fmaxf(ax, bx), tmax);
    tmin = fmaxf(fminf(ay, by), tmin);
    tmax = fminf(fmaxf(ay, by), tmax);
    tmin = fmaxf(fminf(az, bz), tmin);
    tmax = fminf(fmaxf(az, bz), tmax);
    t_entry = tmin;
    return !(tmax <= tmin);
}

// ---------------------------------------------------------------------------------------------
// Sphere::hit, distance only (src/hittable.rs:65-95): half-b quadratic, a = |d|^2 (directions are
// never normalised), strict tmin < t < tmax, near root first.
// ---------------------------------------------------------------------------------------------
// The fast build must not contract these products into FMAs.  c = |oc|^2 - r^2 cancels catastrophically
// when the sphere is far from the origin relative to its radius (10^6-sphere scene: |oc| ~ 300, r = 0.2),
// so whether a scattered ray re-hits the sphere it left ("acne" beyond tmin) depends on the exact
// rounding of oc, |oc|^2 and of the hit point: with contraction the fast build traced 4.4 % more
// segments per path than the reference's arithmetic and rendered that scene 1.5 % darker (measured,
// scripts/dbg_stress_rays.py).  __fmul_rn / __fadd_rn are never contracted; the order is the reference's.
VKD float dot3_rn(float3 a, float3 b) { return __fadd_rn(__fadd_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)), __fmul_rn(a.z, b.z)); }
VKD bool sphere_t(float3 c, float radius, float3 o, float3 d, float tmin, float tmax, float& t) {
    const float3 oc = o - c;
    const float a = dot3_rn(d, d);
    const float half_b = dot3_rn(oc, d);
    const float cc = __fadd_rn(dot3_rn(oc, oc), -__fmul_rn(radius, radius));
    const float disc = __fadd_rn(__fmul_rn(half_b, half_b), -__fmul_rn(a, cc));
    if (disc > 0.0f) {
        const float root = sqrtf(disc);
        float temp = (-half_b - root) / a;
        if (tmin < temp && temp < tmax) {
            t = temp;
            return true;
        }
        temp = (-half_b + root) / a;
        if (tmin < temp && temp < tmax) {
            t = temp;
            return true;
        }
    }
    return false;
}
VKD float3 msphere_center(float4 m0, float4 m1, float time1, float time) { // src/hittable.rs:147-150
    const float3 c0 = f3(m0), c1 = f3(m1);
    return c0 + (c1 - c0) * ((time - m1.w) / (time1 - m1.w));
}

// ---------------------------------------------------------------------------------------------
// Rect::hit, distance only (src/hittable.rs:230-239): inclusive bounds written as the reference
// writes them, so NaN t / NaN a,b pass exactly where they pass there (Q14).
// ---------------------------------------------------------------------------------------------
VKD bool rect_t(float4 bounds, float k, uint32_t axes, float3 o, float3 d, float3 inv_d, float tmin, float tmax, float& t) {
    const uint32_t a0 = axes & 3u, a1 = (axes >> 2) & 3u, a2 = (axes >> 4) & 3u;
#if VK_STRICT
    (void)inv_d;
    const float tt = (k - comp(o, a2)) / comp(d, a2);
#else
    const float tt = (k - comp(o, a2)) * comp(inv_d, a2);
#endif
    if (tt < tmin || tt > tmax) return false;
    const float a = comp(o, a0) + tt * comp(d, a0);
    const float b = comp(o, a1) + tt * comp(d, a1);
    if (a < bounds.x || a > bounds.y || b < bounds.z || b > bounds.w) return false;
    t = tt;
    return true;
}

// ---------------------------------------------------------------------------------------------
// Boxy::hit (src/hittable.rs:363-365) = list hit (:381-394) over the six sides in Boxy::new order
// (:325-353): first side wins ties (strict rec.t < closest_dist), tmax shrinks as sides hit.
// ---------------------------------------------------------------------------------------------
#if !VK_STRICT
// Render build: the same closest side by the slab method.  A ray from outside enters through the FARTHEST of its
// three near planes (that point lies inside the other two slabs, i.e. inside that side's bounds -- the only side
// whose rect test passes before the exit side's), a ray from inside (near planes behind tmin) leaves through the
// NEAREST far plane.  Distances are the rect test's own (k - o) * (1/d), evaluated as one fma each; the list's
// acceptance window is tmin <= t < tmax (the first accepted side needs `rec.t < closest_dist`, :385-389); ties go to
// the side that comes first in Boxy::new order (z, then y, then x).  6 fma + 10 min/max + selects instead of six
// rect tests of ~11 instructions each.
VKD bool box_t(float3 mn, float3 mx, float3 o, float3 d, float3 inv_d, float tmin, float tmax, float& t_out, uint32_t& face) {
    (void)d;
    const float3 oi = f3(-o.x * inv_d.x, -o.y * inv_d.y, -o.z * inv_d.z);
    const float x0 = fmaf(mn.x, inv_d.x, oi.x), x1 = fmaf(mx.x, inv_d.x, oi.x);
    const float y0 = fmaf(mn.y, inv_d.y, oi.y), y1 = fmaf(mx.y, inv_d.y, oi.y);
    const float z0 = fmaf(mn.z, inv_d.z, oi.z), z1 = fmaf(mx.z, inv_d.z, oi.z);
    const float nx = fminf(x0, x1), ny = fminf(y0, y1), nz = fminf(z0, z1);
    const float fx = fmaxf(x0, x1), fy = fmaxf(y0, y1), fz = fmaxf(z0, z1);
    const float t_near = fmaxf(fmaxf(nx, ny), nz), t_far = fminf(fminf(fx, fy), fz);
    if (!(t_near <= t_far)) return false;
    const bool enter = t_near >= tmin;
    const float t = enter ? t_near : t_far;
    if (!(t >= tmin && t < tmax)) return false;
    // which side: the axis that produced t (z, y, x in Boxy::new order), and on it the min or the max plane
    const float cz = enter ? nz : fz, cy = enter ? ny : fy;
    uint32_t axis_face, at_max; // face = 2 * {z: 0, y: 1, x: 2} + (min plane ? 1 : 0)
    if (cz == t) {
        axis_face = 0u;
        at_max = z1 == t;
    } else if (cy == t) {
        axis_face = 2u;
        at_max = y1 == t;
    } else {
        axis_face = 4u;
        at_max = x1 == t;
    }
    t_out = t;
    face = axis_face + (at_max ? 0u : 1u);
    return true;
}
#else
VKD bool box_t(float3 mn, float3 mx, float3 o, float3 d, float3 inv_d, float tmin, float tmax, float& t_out, uint32_t& face) {
    float closest = tmax;
    int f = -1;
#if VK_STRICT
    (void)inv_d;
#define VK_DIV(N, D, I) ((N) / (D))
#else
#define VK_DIV(N, D, I) ((N) * (I))
#endif
#define VK_SIDE(F, K, O2, D2, I2, O0, D0, C0, C1, O1, D1, E0, E1)                                                      \
    {                                                                                                                  \
        const float tt = VK_DIV((K) - (O2), D2, I2);                                                                   \
        if (!(tt < tmin || tt > closest)) {                                                                            \
            const float a = (O0) + tt * (D0), b = (O1) + tt * (D1);                                                    \
            if (!(a < (C0) || a > (C1) || b < (E0) || b > (E1)) && tt < closest) {                                     \
                closest = tt;                                                                                          \
                f = (F);                                                                                               \
            }                                                                                                          \
        }                                                                                                              \
    }
    VK_SIDE(0, mx.z, o.z, d.z, inv_d.z, o.x, d.x, mn.x, mx.x, o.y, d.y, mn.y, mx.y) // XYRect at p1.z
    VK_SIDE(1, mn.z, o.z, d.z, inv_d.z, o.x, d.x, mn.x, mx.x, o.y, d.y, mn.y, mx.y) // FlipFace(XYRect at p0.z)
    VK_SIDE(2, mx.y, o.y, d.y, inv_d.y, o.x, d.x, mn.x, mx.x, o.z, d.z, mn.z, mx.z) // XZRect at p1.y
    VK_SIDE(3, mn.y, o.y, d.y, inv_d.y, o.x, d.x, mn.x, mx.x, o.z, d.z, mn.z, mx.z) // FlipFace(XZRect at p0.y)
    VK_SIDE(4, mx.x, o.x, d.x, inv_d.x, o.y, d.y, mn.y, mx.y, o.z, d.z, mn.z, mx.z) // YZRect at p1.x
    VK_SIDE(5, mn.x, o.x, d.x, inv_d.x, o.y, d.y, mn.y, mx.y, o.z, d.z, mn.z, mx.z) // FlipFace(YZRect at p0.x)
#undef VK_SIDE
#undef VK_DIV
    if (f < 0) return false;
    t_out = closest;
    face = (uint32_t)f;
    return true;
}

#endif
// ---------------------------------------------------------------------------------------------
// Translate / RotateY / RotateX / RotateZ / FlipFace: world -> object ray
// (src/hittable.rs:508, :591-595, :680-684, :769-773) and object -> world point/normal
// (:511, :603-607, :692-696, :781-785).
// ---------------------------------------------------------------------------------------------
VKD void rot_fwd(uint32_t kind, float s, float c, float3& q) {
    const float3 v = q;
    if (kind == VK_X_ROTATE_Y) {
        q.x = c * v.x - s * v.z;
        q.z = s * v.x + c * v.z;
    } else if (kind == VK_X_ROTATE_X) {
        q.y = c * v.y + s * v.z;
        q.z = -s * v.y + c * v.z;
    } else if (kind == VK_X_ROTATE_Z) {
        q.x = c * v.x + s * v.y;
        q.y = -s * v.x + c * v.y;
    }
}
VKD void rot_back(uint32_t kind, float s, float c, float3& q) {
    const float3 v = q;
    if (kind == VK_X_ROTATE_Y) {
        q.x = c * v.x + s * v.z;
        q.z = -s * v.x + c * v.z;
    } else if (kind == VK_X_ROTATE_X) {
        q.y = c * v.y - s * v.z;
        q.z = s * v.y + c * v.z;
    } else if (kind == VK_X_ROTATE_Z) {
        q.x = c * v.x - s * v.y;
        q.y = s * v.x + c * v.y;
    }
}
// Walk a wrapper chain down to its first non-wrapper child, transforming the ray on the way.
VKD uint32_t chain_down(const DScene& sc, uint32_t ref, float3& o, float3& d) {
#pragma unroll 1
    while (VKD_TYPE(ref) == VK_T_XFORM) {
        const float4 x0 = __ldg(&sc.xforms[2 * VKD_INDEX(ref)]);
        const float4 x1 = __ldg(&sc.xforms[2 * VKD_INDEX(ref) + 1]);
        const uint32_t kind = __float_as_uint(x0.x);
        if (kind == VK_X_TRANSLATE) {
            o = o - f3(x1);
        } else if (kind != VK_X_FLIP) {
            rot_fwd(kind, x1.x, x1.y, o);
            rot_fwd(kind, x1.x, x1.y, d);
        }
        ref = __float_as_uint(x0.y);
    }
    return ref;
}

// Distance-only hit of a leaf primitive (no BVH below it): the shared body of the traversal's
// leaf test and of ConstantMedium's two boundary queries.
#if VK_STRICT
VKD float3 rcp3(float3 d) { return f3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z); }
#else
// one MUFU.RCP per component (1/+-0 = +-inf as the slab and plane tests need; a denormal component
// flushes to 0 -> inf, where the exact quotient would overflow anyway)
VKD float fast_rcp(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
VKD float3 rcp3(float3 d) { return f3(fast_rcp(d.x), fast_rcp(d.y), fast_rcp(d.z)); }
#endif

VKD bool leaf_t(const DScene& sc, uint32_t ref, float3 o, float3 d, float3 inv_d, float time, float tmin, float tmax, float& t,
                uint32_t& face) {
    const uint32_t i = VKD_INDEX(ref);
    face = 0;
    switch (VKD_TYPE(ref)) {
    case VK_T_SPHERE: {
        const float4 s = __ldg(&sc.spheres[i]);
        return sphere_t(f3(s), s.w, o, d, tmin, tmax, t);
    }
    case VK_T_MSPHERE: {
        const float4 m0 = __ldg(&sc.mspheres[3 * i]), m1 = __ldg(&sc.mspheres[3 * i + 1]), m2 = __ldg(&sc.mspheres[3 * i + 2]);
        return sphere_t(msphere_center(m0, m1, m2.x, time), m0.w, o, d, tmin, tmax, t);
    }
    case VK_T_RECT: {
        const float4 r0 = __ldg(&sc.rects[2 * i]), r1 = __ldg(&sc.rects[2 * i + 1]);
        return rect_t(r0, r1.x, __float_as_uint(r1.y), o, d, inv_d, tmin, tmax, t);
    }
    case VK_T_BOX: {
        const float4 b0 = __ldg(&sc.boxes[2 * i]), b1 = __ldg(&sc.boxes[2 * i + 1]);
        return box_t(f3(b0), f3(b1), o, d, inv_d, tmin, tmax, t, face);
    }
    default: return false;
    }
}

#ifndef VKD_MEDIUM_SPAN
#define VKD_MEDIUM_SPAN 1 // (0: the reference's two boundary queries as two calls, in the render build too -- A/B only)
#endif
// ConstantMedium::hit (src/hittable.rs:453-493).  The boundary is a leaf, possibly behind a wrapper
// chain (t is invariant under the chain).
// (out of line; MediumXi by value so that the callers' copies stay in registers)
static __device__ __noinline__ bool medium_t(const DScene& sc, uint32_t ref, float3 o, float3 d, float time, float tmin, float tmax,
                                      const MediumXi xi, float& t) {
    const float4 m = __ldg(&sc.media[VKD_INDEX(ref)]);
    float3 bo = o, bd = d;
    float t1 = 0.0f, t2 = 0.0f;
#if VK_STRICT || !VKD_MEDIUM_SPAN
    const uint32_t b = chain_down(sc, __float_as_uint(m.x), bo, bd);
    const float3 binv = rcp3(bd);
#else
    // Render build: the boundary's wrapper chain is one affine map composed at upload (Relayout::media_plan), and for a
    // box or sphere boundary BOTH queries -- rec1 = boundary.hit(-inf, inf), rec2 = boundary.hit(rec1.t + 0.0001, inf)
    // -- come from ONE evaluation of the slabs / the quadratic: the two calls compute the same six plane distances (the
    // same two roots) and differ only in which of them their window accepts, so the window logic is replayed on shared
    // values.  Same arithmetic as box_t / sphere_t, same results as calling them twice.
    const float4* mp = sc.media_plan + 4u * VKD_INDEX(ref);
    const float4 mp3 = __ldg(mp + 3);
    const uint32_t b = __float_as_uint(mp3.x);
    if (__float_as_uint(mp3.y)) {
        const float4 r0 = __ldg(mp), r1 = __ldg(mp + 1), r2 = __ldg(mp + 2);
        bo = f3(fmaf(r0.x, o.x, fmaf(r0.y, o.y, fmaf(r0.z, o.z, r0.w))), fmaf(r1.x, o.x, fmaf(r1.y, o.y, fmaf(r1.z, o.z, r1.w))),
                fmaf(r2.x, o.x, fmaf(r2.y, o.y, fmaf(r2.z, o.z, r2.w))));
        bd = f3(fmaf(r0.x, d.x, fmaf(r0.y, d.y, r0.z * d.z)), fmaf(r1.x, d.x, fmaf(r1.y, d.y, r1.z * d.z)),
                fmaf(r2.x, d.x, fmaf(r2.y, d.y, r2.z * d.z)));
    }
    const float3 binv = rcp3(bd);
    bool spanned = false;
    if (VKD_TYPE(b) == VK_T_BOX) {
        const float4 b0 = __ldg(&sc.boxes[2 * VKD_INDEX(b)]), b1 = __ldg(&sc.boxes[2 * VKD_INDEX(b) + 1]);
        const float3 oi = f3(-bo.x * binv.x, -bo.y * binv.y, -bo.z * binv.z);
        const float x0 = fmaf(b0.x, binv.x, oi.x), x1 = fmaf(b1.x, binv.x, oi.x);
        const float y0 = fmaf(b0.y, binv.y, oi.y), y1 = fmaf(b1.y, binv.y, oi.y);
        const float z0 = fmaf(b0.z, binv.z, oi.z), z1 = fmaf(b1.z, binv.z, oi.z);
        const float t_near = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fminf(z0, z1));
        const float t_far = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fmaxf(z0, z1));
        if (!(t_near <= t_far)) return false;
        // box_t(tmin, tmax = inf): t = (t_near >= tmin) ? t_near : t_far, accepted when tmin <= t < inf
        t1 = (t_near >= -CUDART_INF_F) ? t_near : t_far;
        if (!(t1 >= -CUDART_INF_F && t1 < CUDART_INF_F)) return false;
        const float lo = t1 + 0.0001f;
        t2 = (t_near >= lo) ? t_near : t_far;
        if (!(t2 >= lo && t2 < CUDART_INF_F)) return false;
        spanned = true;
    } else if (VKD_TYPE(b) == VK_T_SPHERE) {
        const float4 sp = __ldg(&sc.spheres[VKD_INDEX(b)]);
        const float3 oc = bo - f3(sp);
        const float a = dot3_rn(bd, bd);
        const float half_b = dot3_rn(oc, bd);
        const float cc = __fadd_rn(dot3_rn(oc, oc), -__fmul_rn(sp.w, sp.w));
        const float disc = __fadd_rn(__fmul_rn(half_b, half_b), -__fmul_rn(a, cc));
        if (!(disc > 0.0f)) return false;
        const float root = sqrtf(disc);
        const float ra = (-half_b - root) / a, rb = (-half_b + root) / a;
        // sphere_t(tmin, tmax = inf): the near root if tmin < it < inf, else the far root under the same test
        if (-CUDART_INF_F < ra && ra < CUDART_INF_F) t1 = ra;
        else if (-CUDART_INF_F < rb && rb < CUDART_INF_F) t1 = rb;
        else return false;
        const float lo = t1 + 0.0001f;
        if (lo < ra && ra < CUDART_INF_F) t2 = ra;
        else if (lo < rb && rb < CUDART_INF_F) t2 = rb;
        else return false;
        spanned = true;
    }
    if (!spanned)
#endif
    {
        uint32_t face;
        float lo = -CUDART_INF_F;
#pragma unroll 1
        for (int q = 0; q < 2; ++q) { // rec1 = boundary.hit(-inf, inf); rec2 = boundary.hit(rec1.t + 0.0001, inf)
            float tq;
            if (!leaf_t(sc, b, bo, bd, binv, time, lo, CUDART_INF_F, tq, face)) return false;
            if (q == 0) {
                t1 = tq;
                lo = tq + 0.0001f;
            } else
                t2 = tq;
        }
    }
    if (t1 < tmin) t1 = tmin;
    if (t2 > tmax) t2 = tmax;
    if (t1 >= t2) return false;
    if (t1 < 0.0f) t1 = 0.0f;
    const float ray_length = sqrtf(length2(d));
    const float distance_inside_boundary = (t2 - t1) * ray_length;
    const float hit_distance = m.y * logf(xi.get(VKD_INDEX(ref), (ref & VKD_DUP) ? 1u : 0u));
    if (hit_distance > distance_inside_boundary) return false;
    t = t1 + hit_distance / ray_length;
    return true;
}

// ---------------------------------------------------------------------------------------------
// BVHNode::hit (src/accel.rs:58-83) as a while-while loop over the wide nodes.
//
// The reference recurses left-then-right and prunes the right subtree with tmax = left.t.  The
// closest hit does not depend on the visiting order (ties excepted), so the GPU (i) tests the
// boxes of both children at the parent, (ii) descends into the nearer box first and (iii) keeps
// every lane of a warp in the node loop until it has a primitive to test, then lets all lanes
// test their primitives together.  Any hit a primitive returns replaces the current one, which
// is the reference's tie rule (`l.t < r.t ? left : right`) for left-then-right order.  Only
// (t, primitive, instance) are tracked; the HitRec is built once, after the loop (resolve_hit).
// ---------------------------------------------------------------------------------------------
struct TraceHit {
    float t;
    uint32_t prim; // leaf ref, VK_REF_NONE = miss
    uint32_t inst; // outermost wrapper of the chain the leaf was reached through, or 0
    uint32_t face;
};
#define VKD_DONE 0xFFFFFFFFu

struct TraceCounters {
    uint32_t nodes, prims;
};

// The traversal as a resumable state machine: one call of trav_node_step / trav_prim_step advances
// one lane by one node visit / one primitive test.  trace() below runs it to completion for one ray
// (while-while); the dynamic megakernel (vk_kernels.cu) interleaves steps of all the lanes of a warp
// under warp votes and leaves the loop to re-fill idle lanes.
struct Trav {
    uint32_t stack[VKD_STACK];
    int sp;
    float3 co, cd, cinv; // ray in the current frame (world, or the frame of the instance being traversed)
    uint32_t cur_inst;
    uint32_t ref;  // what to process next; VKD_DONE when the traversal has finished
    bool enter;    // `ref` is a BVH root whose own box has not been tested yet
    TraceHit best;
};
VKD void trav_init(Trav& T, const DScene& sc, float3 o, float3 d, float tmax) {
    T.sp = 0;
    T.co = o;
    T.cd = d;
    T.cinv = rcp3(d);
    T.cur_inst = 0;
    T.best.t = tmax;
    T.best.prim = VK_REF_NONE;
    T.best.inst = 0;
    T.best.face = 0;
    T.ref = sc.root;
    T.enter = true;
}
VKD uint32_t trav_pop(Trav& T) { return T.sp ? T.stack[--T.sp] : VKD_DONE; }
VKD bool trav_at_node(const Trav& T) { return T.ref != VKD_DONE && VKD_TYPE(T.ref) == VK_T_NODE; }
// One visit of a four-wide node: the four AxisBB::hit tests and the hits sorted by entry distance (r0 nearest; a missed
// or empty slot is VK_REF_NONE and sorts last).  Shared by the lane traversal (Trav, stack in local memory) and the
// step-queue kernel (vk_stepq.cu, stack in shared memory).
VKD void wide_node_test(const DScene& sc, uint32_t ni, float3 co, float3 cd, float3 cinv, float tmin, float tmax, uint32_t& r0, uint32_t& r1,
                        uint32_t& r2, uint32_t& r3) {
    const float4* w = sc.wnodes + 8u * (size_t)ni;
    const float4 mnx = __ldg(w), mxx = __ldg(w + 1), mny = __ldg(w + 2), mxy = __ldg(w + 3), mnz = __ldg(w + 4), mxz = __ldg(w + 5);
    const float4 rf = __ldg(w + 6);
    r0 = __float_as_uint(rf.x), r1 = __float_as_uint(rf.y), r2 = __float_as_uint(rf.z), r3 = __float_as_uint(rf.w);
    float t0, t1, t2, t3;
    // AxisBB::hit per slot (src/accel.rs:16-35); a missed or empty slot drops out (ref 0, t = +inf)
#if VK_STRICT
    if (!(r0 != VK_REF_NONE && aabb_hit(f3(mnx.x, mny.x, mnz.x), f3(mxx.x, mxy.x, mxz.x), co, cd, cinv, tmin, tmax, t0))) { r0 = VK_REF_NONE; t0 = CUDART_INF_F; }
    if (!(r1 != VK_REF_NONE && aabb_hit(f3(mnx.y, mny.y, mnz.y), f3(mxx.y, mxy.y, mxz.y), co, cd, cinv, tmin, tmax, t1))) { r1 = VK_REF_NONE; t1 = CUDART_INF_F; }
    if (!(r2 != VK_REF_NONE && aabb_hit(f3(mnx.z, mny.z, mnz.z), f3(mxx.z, mxy.z, mxz.z), co, cd, cinv, tmin, tmax, t2))) { r2 = VK_REF_NONE; t2 = CUDART_INF_F; }
    if (!(r3 != VK_REF_NONE && aabb_hit(f3(mnx.w, mny.w, mnz.w), f3(mxx.w, mxy.w, mxz.w), co, cd, cinv, tmin, tmax, t3))) { r3 = VK_REF_NONE; t3 = CUDART_INF_F; }
#else
    {   // the same slab test with one FMA per plane: (b - o) * (1/d) = b * (1/d) - o * (1/d)
        const float3 oi = f3(-co.x * cinv.x, -co.y * cinv.y, -co.z * cinv.z);
#define VKD_SLAB(C, R, TO)                                                                                             \
        {                                                                                                              \
            const float ax = fmaf(mnx.C, cinv.x, oi.x), bx = fmaf(mxx.C, cinv.x, oi.x);                            \
            const float ay = fmaf(mny.C, cinv.y, oi.y), by = fmaf(mxy.C, cinv.y, oi.y);                            \
            const float az = fmaf(mnz.C, cinv.z, oi.z), bz = fmaf(mxz.C, cinv.z, oi.z);                            \
            const float tn = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fmaxf(fminf(az, bz), tmin));                   \
            const float tf = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fminf(fmaxf(az, bz), tmax));                   \
            const bool miss = (R == VK_REF_NONE) | (tf <= tn);                                                         \
            TO = miss ? CUDART_INF_F : tn;                                                                             \
            R = miss ? VK_REF_NONE : R;                                                                                \
        }
        VKD_SLAB(x, r0, t0)
        VKD_SLAB(y, r1, t1)
        VKD_SLAB(z, r2, t2)
        VKD_SLAB(w, r3, t3)
#undef VKD_SLAB
    }
#endif
    // sort the four (t, ref) pairs by entry distance: 5-comparator network, misses sink to the end
#define VKD_CSWAP(TA, RA, TB, RB)                                                                                      \
    {                                                                                                                  \
        const bool sw = TB < TA;                                                                                       \
        const float tt_ = sw ? TA : TB;                                                                                \
        const uint32_t rr_ = sw ? RA : RB;                                                                             \
        TA = sw ? TB : TA;                                                                                             \
        RA = sw ? RB : RA;                                                                                             \
        TB = tt_;                                                                                                      \
        RB = rr_;                                                                                                      \
    }
    VKD_CSWAP(t0, r0, t1, r1)
    VKD_CSWAP(t2, r2, t3, r3)
    VKD_CSWAP(t0, r0, t2, r2)
    VKD_CSWAP(t1, r1, t3, r3)
    VKD_CSWAP(t1, r1, t2, r2)
#undef VKD_CSWAP
}
// precondition: trav_at_node(T)
VKD void trav_node_step(Trav& T, const DScene& sc, float tmin, TraceCounters& tc) {
    const uint32_t ni = VKD_INDEX(T.ref);
    if (T.enter) { // BVHNode::hit's own `bb.hit` for the world root / an instanced sub-BVH root
        T.enter = false;
        const float4 n0 = __ldg(&sc.nodes[2 * ni]), n1 = __ldg(&sc.nodes[2 * ni + 1]);
        float te;
        if (!aabb_hit(f3(n0), f3(n1), T.co, T.cd, T.cinv, tmin, T.best.t, te)) {
            T.ref = trav_pop(T);
            return;
        }
    }
    ++tc.nodes;
    uint32_t r0, r1, r2, r3;
    wide_node_test(sc, ni, T.co, T.cd, T.cinv, tmin, T.best.t, r0, r1, r2, r3);
    // nearest first, the others wait on the stack, farthest deepest
    if (r3 != VK_REF_NONE) T.stack[T.sp++] = r3;
    if (r2 != VK_REF_NONE) T.stack[T.sp++] = r2;
    if (r1 != VK_REF_NONE) T.stack[T.sp++] = r1;
    T.ref = r0 != VK_REF_NONE ? r0 : trav_pop(T);
}
// precondition: T.ref is neither VKD_DONE nor a node; (o, d) is the world ray
template <bool MEDIA>
VKD void trav_prim_step(Trav& T, const DScene& sc, float3 o, float3 d, float time, float tmin, const MediumXi& xi, TraceCounters& tc) {
    const uint32_t ref = T.ref;
    const uint32_t type = VKD_TYPE(ref);
    if (type == VKD_T_EXIT) { // leave the instanced sub-BVH
        T.co = o;
        T.cd = d;
        T.cinv = rcp3(d);
        T.cur_inst = 0;
    } else if (type != VK_T_NONE) {
        float3 to = T.co, td = T.cd, tinv = T.cinv;
        uint32_t leaf = ref, inst = T.cur_inst;
        if (type == VK_T_XFORM) {
            leaf = chain_down(sc, ref, to, td) | (ref & VKD_DUP);
            inst = ref & ~VKD_DUP;
            if (VKD_TYPE(leaf) == VK_T_NODE) { // instanced sub-BVH: traverse it in object space
                T.stack[T.sp++] = VKD_T_EXIT << 28;
                T.co = to;
                T.cd = td;
                T.cinv = rcp3(td);
                T.cur_inst = inst;
                T.ref = leaf & ~VKD_DUP;
                T.enter = true;
                return;
            }
            tinv = rcp3(td);
        }
        float t;
        uint32_t face = 0;
        bool hit;
        ++tc.prims;
        if (MEDIA && VKD_TYPE(leaf) == VK_T_MEDIUM) hit = medium_t(sc, leaf, to, td, time, tmin, T.best.t, xi, t);
        else hit = leaf_t(sc, leaf, to, td, tinv, time, tmin, T.best.t, t, face);
        if (hit) {
            T.best.t = t;
            T.best.prim = leaf & ~VKD_DUP;
            T.best.inst = inst;
            T.best.face = face;
        }
    }
    T.ref = trav_pop(T);
}

template <bool MEDIA>
VKD TraceHit trace(const DScene& sc, float3 o, float3 d, float time, float tmin, float tmax, const MediumXi& xi, TraceCounters& tc) {
    Trav T;
    trav_init(T, sc, o, d, tmax);
#pragma unroll 1
    for (;;) {
#pragma unroll 1
        while (trav_at_node(T)) trav_node_step(T, sc, tmin, tc); // every lane stays here until it holds a primitive
        if (T.ref == VKD_DONE) break;
        trav_prim_step<MEDIA>(T, sc, o, d, time, tmin, xi, tc); // then all lanes test their primitives together
    }
    return T.best;
}

// ---------------------------------------------------------------------------------------------
// The same closest-hit query over a flat program (see FlatProgram in vk_internal.h): typed batches,
// every lane runs the same entry at the same time.  Per-entry arithmetic is the reference's, in
// its order (STRICT divides, FAST multiplies by 1/d).
// ---------------------------------------------------------------------------------------------
#if VK_STRICT
#define VKF_PLANE_T(K, O, D, I) (((K) - (O)) / (D))
#else
#define VKF_PLANE_T(K, O, D, I) (((K) - (O)) * (I))
#endif
// AX: 0 = XYRect (plane on z), 1 = XZRect (plane on y), 2 = YZRect (plane on x); src/hittable.rs:214-239.
// BOX_SIDE: the entry is a side of a Boxy -- list semantics, strictly closer only (:386).
template <int AX, bool BOX_SIDE>
VKD void flat_rects(const FlatProgram& P, uint32_t i0, uint32_t i1, float3 co, float3 cd, float3 ci, float tmin, float& best_t,
                    uint32_t& best_hit) {
#pragma unroll 1
    for (uint32_t i = i0; i < i1; ++i) {
        const float4 bd = P.rects[i].bounds;
        const float k = P.rects[i].k;
        float tt, a, b;
        if (AX == 0) {
            tt = VKF_PLANE_T(k, co.z, cd.z, ci.z);
            a = co.x + tt * cd.x;
            b = co.y + tt * cd.y;
        } else if (AX == 1) {
            tt = VKF_PLANE_T(k, co.y, cd.y, ci.y);
            a = co.x + tt * cd.x;
            b = co.z + tt * cd.z;
        } else {
            tt = VKF_PLANE_T(k, co.x, cd.x, ci.x);
            a = co.y + tt * cd.y;
            b = co.z + tt * cd.z;
        }
        bool hit = !(tt < tmin || tt > best_t) && !(a < bd.x || a > bd.y || b < bd.z || b > bd.w);
        if (BOX_SIDE) hit = hit && tt < best_t;
        if (hit) {
            best_t = tt;
            best_hit = P.rects[i].hit;
        }
    }
}
#if !VK_STRICT
// Render build: a Boxy of the flat program as ONE entry, by the slab method (box_t above has the argument: a ray from
// outside enters through the farthest of its three near planes, a ray from inside leaves through the nearest far
// plane; acceptance window tmin <= t < best as for a box side, ties to the side that comes first in Boxy::new order).
// The plane distances are the rect test's own (k - o) * (1/d), NOT one fma each: a ray that starts on a side keeps the
// exact t = 0 it has in the six-rect form (see the rejected experiment in flat_rects_k).  ~40 instructions per ray
// instead of six rect tests of ~15.  The winning side's entry of the hit table: sides 0|1, 2|3, 4|5 are consecutive.
template <int K>
VKD void flat_box_k(const FlatBox& bx, const float3 (&co)[K], const float3 (&ci)[K], float tmin, float (&best_t)[K], uint32_t (&best_hit)[K]) {
    const float4 mn = bx.mn, mx = bx.mx;
    const uint32_t hz = __float_as_uint(mn.w), hy = __float_as_uint(mx.w) & 0xFFFFu, hx = __float_as_uint(mx.w) >> 16;
#pragma unroll
    for (int q = 0; q < K; ++q) {
        const float x0 = (mn.x - co[q].x) * ci[q].x, x1 = (mx.x - co[q].x) * ci[q].x;
        const float y0 = (mn.y - co[q].y) * ci[q].y, y1 = (mx.y - co[q].y) * ci[q].y;
        const float z0 = (mn.z - co[q].z) * ci[q].z, z1 = (mx.z - co[q].z) * ci[q].z;
        const float nx = fminf(x0, x1), ny = fminf(y0, y1), nz = fminf(z0, z1);
        const float fx = fmaxf(x0, x1), fy = fmaxf(y0, y1), fz = fmaxf(z0, z1);
        const float t_near = fmaxf(fmaxf(nx, ny), nz), t_far = fminf(fminf(fx, fy), fz);
        const bool enter = t_near >= tmin;
        const float t = enter ? t_near : t_far;
        const bool hit = (t_near <= t_far) & (t >= tmin) & (t < best_t[q]);
        const bool on_z = (enter ? nz : fz) == t, on_y = (enter ? ny : fy) == t;
        const float at_max = on_z ? z1 : (on_y ? y1 : x1); // distance of the axis' box_max plane: sides 0, 2, 4
        const uint32_t id = (on_z ? hz : (on_y ? hy : hx)) + (at_max == t ? 0u : 1u);
        best_t[q] = hit ? t : best_t[q];
        best_hit[q] = hit ? id : best_hit[q];
    }
}
template <int K>
VKD void flat_boxes_k(const FlatProgram& P, uint32_t i0, uint32_t i1, const float3 (&co)[K], const float3 (&ci)[K], float tmin,
                      float (&best_t)[K], uint32_t (&best_hit)[K]) {
#pragma unroll 1
    for (uint32_t i = i0; i < i1; ++i) flat_box_k<K>(P.boxes[i], co, ci, tmin, best_t, best_hit);
}
#endif
template <bool MEDIA>
VKD TraceHit trace_flat(const DScene& sc, const FlatProgram& P, float3 o, float3 d, float time, float tmin, float tmax,
                        const MediumXi& xi, TraceCounters& tc) {
    float best_t = tmax;
    uint32_t best_hit = 0xFFFFFFFFu;
    TraceHit sub; // closest hit inside a subtree of a hybrid program
    sub.t = tmax;
    sub.prim = VK_REF_NONE;
    sub.inst = 0;
    sub.face = 0;
    const uint32_t n_segs = P.n_segs;
    tc.prims += P.n;
#pragma unroll 1
    for (uint32_t s = 0; s < n_segs; ++s) {
        const FlatSeg& g = P.segs[s];
        float3 co = o, cd = d;
#pragma unroll 1
        for (uint32_t k = g.op0; k < g.op1; ++k) { // world ray -> frame of this instance chain
            const uint32_t kind = P.ops[k].kind;
            if (kind == VKF_OP_TRANSLATE) co = co - f3(P.ops[k].a, P.ops[k].b, P.ops[k].c);
            else {
                rot_fwd(kind, P.ops[k].a, P.ops[k].b, co); // VKF_OP_ROT* == VK_X_ROTATE_*
                rot_fwd(kind, P.ops[k].a, P.ops[k].b, cd);
            }
        }
        const float3 ci = rcp3(cd);
        flat_rects<0, false>(P, g.rect0[0], g.rect1[0], co, cd, ci, tmin, best_t, best_hit);
        flat_rects<1, false>(P, g.rect0[1], g.rect1[1], co, cd, ci, tmin, best_t, best_hit);
        flat_rects<2, false>(P, g.rect0[2], g.rect1[2], co, cd, ci, tmin, best_t, best_hit);
#if VK_STRICT
        flat_rects<0, true>(P, g.rect0[3], g.rect1[3], co, cd, ci, tmin, best_t, best_hit);
        flat_rects<1, true>(P, g.rect0[4], g.rect1[4], co, cd, ci, tmin, best_t, best_hit);
        flat_rects<2, true>(P, g.rect0[5], g.rect1[5], co, cd, ci, tmin, best_t, best_hit);
#else
        {
            const float3 co1[1] = {co}, ci1[1] = {ci};
            float bt1[1] = {best_t};
            uint32_t bh1[1] = {best_hit};
            flat_boxes_k<1>(P, g.box0, g.box1, co1, ci1, tmin, bt1, bh1);
            best_t = bt1[0];
            best_hit = bh1[0] == 0xFFFFFFFFu ? bh1[0] : VKF_HIT_INDEX(bh1[0]); // (the box entries carry class-tagged ids)
        }
#endif
#pragma unroll 1
        for (uint32_t i = g.sph0; i < g.sph1; ++i) {
            float tt;
            if (sphere_t(f3(P.spheres[i].a), P.spheres[i].a.w, co, cd, tmin, best_t, tt)) {
                best_t = tt;
                best_hit = P.spheres[i].hit;
            }
        }
#pragma unroll 1
        for (uint32_t i = g.msph0; i < g.msph1; ++i) {
            float tt;
            if (sphere_t(msphere_center(P.spheres[i].a, P.spheres[i].b, P.spheres[i].time1, time), P.spheres[i].a.w, co, cd, tmin, best_t, tt)) {
                best_t = tt;
                best_hit = P.spheres[i].hit;
            }
        }
        if (MEDIA) {
#pragma unroll 1
            for (uint32_t i = g.med0; i < g.med1; ++i) {
                float tt;
                if (medium_t(sc, P.hits[i].prim, co, cd, time, tmin, best_t, xi, tt)) {
                    best_t = tt;
                    best_hit = i;
                }
            }
        }
        // homogeneous subtrees of a hybrid program: while-while over the 4-wide nodes in this frame
#pragma unroll 1
        for (uint32_t i = g.bvh0; i < g.bvh1; ++i) {
            Trav T;
            T.sp = 0;
            T.co = co;
            T.cd = cd;
            T.cinv = ci;
            T.cur_inst = P.seg_inst[s];
            T.best.t = best_t;
            T.best.prim = VK_REF_NONE;
            T.best.inst = 0;
            T.best.face = 0;
            T.ref = P.bvh[i];
            T.enter = true;
#pragma unroll 1
            for (;;) {
#pragma unroll 1
                while (trav_at_node(T)) trav_node_step(T, sc, tmin, tc);
                if (T.ref == VKD_DONE) break;
                trav_prim_step<false>(T, sc, o, d, time, tmin, xi, tc); // leaves only: no wrapper, no medium below
            }
            if (T.best.prim != VK_REF_NONE) {
                best_t = T.best.t;
                sub = T.best;
                best_hit = 0xFFFFFFFEu;
            }
        }
    }
    TraceHit best;
    best.t = best_t;
    best.prim = VK_REF_NONE;
    best.inst = 0;
    best.face = 0;
    if (best_hit == 0xFFFFFFFEu) return sub; // the closest hit came from a subtree
    if (best_hit != 0xFFFFFFFFu) {
        best.prim = P.hits[best_hit].prim & ~VKD_DUP;
        best.inst = P.hits[best_hit].inst;
        best.face = P.hits[best_hit].face;
    }
    return best;
}

// K rays per thread through the flat program (the staged kernel traces all the slots a thread owns
// together): an entry's operands are fetched once for the K rays and the K closest-hit chains are
// independent, which is the instruction-level parallelism a warp-per-SM-quarter schedule lacks.
// One rect entry for K rays (flat_rects_k walks a range of them, trace_flat_static names each one).
template <int K, int AX, bool BOX_SIDE>
VKD void flat_rect_k(const FlatRect& r, const float3 (&co)[K], const float3 (&cd)[K], const float3 (&ci)[K], float tmin, float (&best_t)[K],
                     uint32_t (&best_hit)[K]) {
    const float4 bd = r.bounds;
    const float k = r.k;
    const uint32_t id = r.hitc;
#pragma unroll
    for (int q = 0; q < K; ++q) {
        float tt, a, b;
        if (AX == 0) {
            tt = VKF_PLANE_T(k, co[q].z, cd[q].z, ci[q].z);
            a = co[q].x + tt * cd[q].x;
            b = co[q].y + tt * cd[q].y;
        } else if (AX == 1) {
            tt = VKF_PLANE_T(k, co[q].y, cd[q].y, ci[q].y);
            a = co[q].x + tt * cd[q].x;
            b = co[q].z + tt * cd[q].z;
        } else {
            tt = VKF_PLANE_T(k, co[q].x, cd[q].x, ci[q].x);
            a = co[q].y + tt * cd[q].y;
            b = co[q].z + tt * cd[q].z;
        }
        // same predicate as Rect::hit, evaluated without branches (bitwise on the comparison results).
        // (Measured and rejected in round 2: the plane distance as one fma, k * (1/d) - o * (1/d), and the bounds as
        // |a - centre| <= half extent.  0.6 % faster, but a ray that STARTS on the plane -- every scattered ray --
        // no longer gets t = 0 exactly: the two products cancel to rounding noise of either sign, scaled by 1/d.
        // Dropped samples rose from 26 to 1503 per 3.6e8 paths and light leaked around the box.)
        // (the comparison with the closest hit so far comes last: it is the only link between one entry and the next)
        bool miss = (a < bd.x) | (a > bd.y) | (b < bd.z) | (b > bd.w) | (tt < tmin);
        miss = miss | (tt > best_t[q]);
        if (BOX_SIDE) miss = miss | !(tt < best_t[q]);
        best_t[q] = miss ? best_t[q] : tt;
        best_hit[q] = miss ? best_hit[q] : id;
    }
}
template <int K, int AX, bool BOX_SIDE>
VKD void flat_rects_k(const FlatProgram& P, uint32_t i0, uint32_t i1, const float3 (&co)[K], const float3 (&cd)[K], const float3 (&ci)[K],
                      float tmin, float (&best_t)[K], uint32_t (&best_hit)[K]) {
    // (unrolled by two, ptxas fetches the operands with per-thread LDC instead of uniform LDCU and the loop grows; the six
    // compares of a ray as three independent two-compare chains joined by one PLOP3 -- depth 3 instead of 6, one more
    // instruction -- is 1 % slower: the loop is bound by what it issues, not by the predicate chain, profiles/r2_sweep_15.log)
#pragma unroll 1
    for (uint32_t i = i0; i < i1; ++i) flat_rect_k<K, AX, BOX_SIDE>(P.rects[i], co, cd, ci, tmin, best_t, best_hit);
}
// `live` masks the rays that exist (an idle slot's ray is traced as a dummy and ignored); best_hit
// is 0xFFFFFFFF or the class-tagged id of the entry (VKF_HITC: index into P.hits | queue class << 8).
// HYBRID: the program may hold homogeneous subtrees (FlatProgram::bvh); a ray whose closest hit came from one gets
// best_hit = 0xFFFFFFFE and the hit itself in sub[] (as in trace_flat).
#if !VK_STRICT
// ConstantMedium::hit for a flat-program entry whose boundary is a Boxy, on operands from the constant bank (FlatMedium):
// medium_t's render-build arithmetic -- the boundary chain as one affine map, both boundary queries replayed on one slab
// evaluation -- without the call, the loads of the medium / plan / box records and the switch on the boundary's type.
#ifndef VKF_INLINE_MEDIA
#define VKF_INLINE_MEDIA 1
#endif
VKD bool flat_medium_box(const FlatMedium& fm, uint32_t ref, float3 o, float3 d, float tmin, float tmax, const MediumXi& xi, float& t) {
    float3 bo = o, bd = d;
    if (__float_as_uint(fm.mx.w) & 2u) {
        const float* m = fm.aff;
        bo = f3(fmaf(m[0], o.x, fmaf(m[1], o.y, fmaf(m[2], o.z, m[9]))), fmaf(m[3], o.x, fmaf(m[4], o.y, fmaf(m[5], o.z, m[10]))),
                fmaf(m[6], o.x, fmaf(m[7], o.y, fmaf(m[8], o.z, m[11]))));
        bd = f3(fmaf(m[0], d.x, fmaf(m[1], d.y, m[2] * d.z)), fmaf(m[3], d.x, fmaf(m[4], d.y, m[5] * d.z)),
                fmaf(m[6], d.x, fmaf(m[7], d.y, m[8] * d.z)));
    }
    const float3 binv = rcp3(bd);
    const float3 oi = f3(-bo.x * binv.x, -bo.y * binv.y, -bo.z * binv.z);
    const float x0 = fmaf(fm.mn.x, binv.x, oi.x), x1 = fmaf(fm.mx.x, binv.x, oi.x);
    const float y0 = fmaf(fm.mn.y, binv.y, oi.y), y1 = fmaf(fm.mx.y, binv.y, oi.y);
    const float z0 = fmaf(fm.mn.z, binv.z, oi.z), z1 = fmaf(fm.mx.z, binv.z, oi.z);
    const float t_near = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fminf(z0, z1));
    const float t_far = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fmaxf(z0, z1));
    if (!(t_near <= t_far)) return false;
    float t1 = (t_near >= -CUDART_INF_F) ? t_near : t_far; // (the window logic of box_t, see medium_t)
    if (!(t1 >= -CUDART_INF_F && t1 < CUDART_INF_F)) return false;
    const float lo = t1 + 0.0001f;
    float t2 = (t_near >= lo) ? t_near : t_far;
    if (!(t2 >= lo && t2 < CUDART_INF_F)) return false;
    if (t1 < tmin) t1 = tmin;
    if (t2 > tmax) t2 = tmax;
    if (t1 >= t2) return false;
    if (t1 < 0.0f) t1 = 0.0f;
    const float ray_length = sqrtf(length2(d));
    const float distance_inside_boundary = (t2 - t1) * ray_length;
    const float hit_distance = fm.mn.w * logf(xi.get(VKD_INDEX(ref), (ref & VKD_DUP) ? 1u : 0u));
    if (hit_distance > distance_inside_boundary) return false;
    t = t1 + hit_distance / ray_length;
    return true;
}
#endif
// One static sphere entry for K rays.
template <int K>
VKD void flat_sphere_k(const FlatSphere& s, const float3 (&co)[K], const float3 (&cd)[K], float tmin, float (&best_t)[K], uint32_t (&best_hit)[K]) {
    const float4 sp = s.a;
    const uint32_t id = s.hitc;
#pragma unroll
    for (int q = 0; q < K; ++q) {
        float tt;
        if (sphere_t(f3(sp), sp.w, co[q], cd[q], tmin, best_t[q], tt)) {
            best_t[q] = tt;
            best_hit[q] = id;
        }
    }
}
// The world rays (wo, wd) into a segment's frame through its chain composed into one affine map m (render build).
template <int K>
VKD void flat_affine_k(const float* m, const float3 (&wo)[K], const float3 (&wd)[K], float3 (&co)[K], float3 (&cd)[K]) {
    const float r00 = m[0], r01 = m[1], r02 = m[2], r10 = m[3], r11 = m[4], r12 = m[5], r20 = m[6], r21 = m[7], r22 = m[8];
    const float t0 = m[9], t1 = m[10], t2 = m[11];
#pragma unroll
    for (int q = 0; q < K; ++q) {
        const float3 o = wo[q], d = wd[q];
        co[q] = f3(fmaf(r00, o.x, fmaf(r01, o.y, fmaf(r02, o.z, t0))), fmaf(r10, o.x, fmaf(r11, o.y, fmaf(r12, o.z, t1))),
                   fmaf(r20, o.x, fmaf(r21, o.y, fmaf(r22, o.z, t2))));
        cd[q] = f3(fmaf(r00, d.x, fmaf(r01, d.y, r02 * d.z)), fmaf(r10, d.x, fmaf(r11, d.y, r12 * d.z)),
                   fmaf(r20, d.x, fmaf(r21, d.y, r22 * d.z)));
    }
}
// One segment of the program: (co, cd) is the ray in the segment's frame, (o, d) the world ray.
template <int K, bool MEDIA, bool HYBRID>
VKD void flat_segment_k(const DScene& sc, const FlatProgram& P, const FlatSeg& g, uint32_t s, const float3 (&o)[K], const float3 (&d)[K],
                        const float3 (&co)[K], const float3 (&cd)[K], const float (&time)[K], const bool (&live)[K], float tmin,
                        const MediumXi (&xi)[K], float (&best_t)[K], uint32_t (&best_hit)[K], TraceHit* sub, TraceCounters* tc) {
    float3 ci[K];
#pragma unroll
    for (int q = 0; q < K; ++q) ci[q] = rcp3(cd[q]);
    flat_rects_k<K, 0, false>(P, g.rect0[0], g.rect1[0], co, cd, ci, tmin, best_t, best_hit);
    flat_rects_k<K, 1, false>(P, g.rect0[1], g.rect1[1], co, cd, ci, tmin, best_t, best_hit);
    flat_rects_k<K, 2, false>(P, g.rect0[2], g.rect1[2], co, cd, ci, tmin, best_t, best_hit);
#if VK_STRICT
    flat_rects_k<K, 0, true>(P, g.rect0[3], g.rect1[3], co, cd, ci, tmin, best_t, best_hit);
    flat_rects_k<K, 1, true>(P, g.rect0[4], g.rect1[4], co, cd, ci, tmin, best_t, best_hit);
    flat_rects_k<K, 2, true>(P, g.rect0[5], g.rect1[5], co, cd, ci, tmin, best_t, best_hit);
#else
    flat_boxes_k<K>(P, g.box0, g.box1, co, ci, tmin, best_t, best_hit);
#endif
#pragma unroll 1
    for (uint32_t i = g.sph0; i < g.sph1; ++i) flat_sphere_k<K>(P.spheres[i], co, cd, tmin, best_t, best_hit);
#if !VK_SIMPLE
#pragma unroll 1
    for (uint32_t i = g.msph0; i < g.msph1; ++i) {
#pragma unroll
        for (int q = 0; q < K; ++q) {
            float tt;
            if (sphere_t(msphere_center(P.spheres[i].a, P.spheres[i].b, P.spheres[i].time1, time[q]), P.spheres[i].a.w, co[q], cd[q], tmin, best_t[q], tt)) {
                best_t[q] = tt;
                best_hit[q] = P.spheres[i].hitc;
            }
        }
    }
#endif
    if (MEDIA) {
#pragma unroll 1
        for (uint32_t i = g.med0; i < g.med1; ++i) {
#if !VK_STRICT && VKF_INLINE_MEDIA
            const FlatMedium& fm = P.fmed[P.seg_fm0[s] + (i - g.med0)];
            const bool inline_box = (__float_as_uint(fm.mx.w) & 1u) != 0u; // (uniform: the constant bank)
#endif
#pragma unroll // (static indices: a rolled loop over q sends co / cd / best_t / xi to local memory for the whole function)
            for (int q = 0; q < K; ++q) {
                float tt;
                bool hit;
#if !VK_STRICT && VKF_INLINE_MEDIA
                if (inline_box) hit = live[q] && flat_medium_box(fm, P.hits[i].prim, co[q], cd[q], tmin, best_t[q], xi[q], tt);
                else
#endif
                    hit = live[q] && medium_t(sc, P.hits[i].prim, co[q], cd[q], time[q], tmin, best_t[q], xi[q], tt);
                if (hit) {
                    best_t[q] = tt;
                    best_hit[q] = VKF_HITC(i, P.hits[i].cls, P.hits[i].inst);
                }
            }
        }
    }
    if (HYBRID) { // homogeneous subtrees: every lane walks the 4-wide nodes for its own ray, in this segment's frame
#pragma unroll 1
        for (uint32_t i = g.bvh0; i < g.bvh1; ++i) {
#pragma unroll
            for (int q = 0; q < K; ++q) {
                Trav T;
                T.sp = 0;
                T.co = co[q];
                T.cd = cd[q];
                T.cinv = ci[q];
                T.cur_inst = P.seg_inst[s];
                T.best.t = best_t[q];
                T.best.prim = VK_REF_NONE;
                T.best.inst = 0;
                T.best.face = 0;
                T.ref = live[q] ? P.bvh[i] : VKD_DONE;
                T.enter = true;
#pragma unroll 1
                for (;;) {
#pragma unroll 1
                    while (trav_at_node(T)) trav_node_step(T, sc, tmin, *tc);
                    if (T.ref == VKD_DONE) break;
                    trav_prim_step<false>(T, sc, o[q], d[q], time[q], tmin, xi[q], *tc); // leaves only: no wrapper, no medium below
                }
                if (T.best.prim != VK_REF_NONE) {
                    best_t[q] = T.best.t;
                    sub[q] = T.best;
                    best_hit[q] = 0xFFFFFFFEu;
                }
            }
        }
    }
}
#ifndef VKF_PEEL_WORLD
#define VKF_PEEL_WORLD 1
#endif
template <int K, bool MEDIA, bool HYBRID = false>
VKD void trace_flat_k(const DScene& sc, const FlatProgram& P, const float3 (&o)[K], const float3 (&d)[K], const float (&time)[K],
                      const bool (&live)[K], float tmin, const MediumXi (&xi)[K], float (&best_t)[K], uint32_t (&best_hit)[K],
                      TraceHit* sub = nullptr, TraceCounters* tc = nullptr) {
#pragma unroll
    for (int q = 0; q < K; ++q) {
        best_t[q] = CUDART_INF_F;
        best_hit[q] = 0xFFFFFFFFu;
    }
    const uint32_t n_segs = P.n_segs;
#if !VK_STRICT && VKF_PEEL_WORLD
    // Segment 0 is the world frame (no ops, FlatBuilder::build): the ray as it is.  Inside the loop the world ray would
    // be copied into the registers the instance segments overwrite, 6 moves per ray and segment (1.9 % of the Cornell
    // kernel's instructions).  Measured (profiles/r2_sweep_17.log): Cornell 32.65 -> 32.53 ms, perlin demo 2.98 -> 2.78 ms;
    // the media kernels LOSE 1.2 % (Cornell smoke 21.56 -> 21.83 ms: one segment, and a second copy of the medium loop
    // for nothing), so they keep the loop below.
    if constexpr (!MEDIA) {
    flat_segment_k<K, MEDIA, HYBRID>(sc, P, P.segs[0], 0u, o, d, o, d, time, live, tmin, xi, best_t, best_hit, sub, tc);
#pragma unroll 1
    for (uint32_t s = 1; s < n_segs; ++s) {
        const FlatSeg& g = P.segs[s];
        float3 co[K], cd[K];
        flat_affine_k<K>(P.seg_affine[s], o, d, co, cd); // the chain as one affine map (composed at upload): no loop, no switch on the wrapper kind
        flat_segment_k<K, MEDIA, HYBRID>(sc, P, g, s, o, d, co, cd, time, live, tmin, xi, best_t, best_hit, sub, tc);
    }
    return;
    }
#endif
    {
#pragma unroll 1
    for (uint32_t s = 0; s < n_segs; ++s) {
        const FlatSeg& g = P.segs[s];
        float3 co[K], cd[K];
#pragma unroll
        for (int q = 0; q < K; ++q) {
            co[q] = o[q];
            cd[q] = d[q];
        }
#if VK_STRICT
#pragma unroll 1
        for (uint32_t k = g.op0; k < g.op1; ++k) {
            const uint32_t kind = P.ops[k].kind;
            const float pa = P.ops[k].a, pb = P.ops[k].b, pc = P.ops[k].c;
#pragma unroll
            for (int q = 0; q < K; ++q) {
                if (kind == VKF_OP_TRANSLATE) co[q] = co[q] - f3(pa, pb, pc);
                else {
                    rot_fwd(kind, pa, pb, co[q]);
                    rot_fwd(kind, pa, pb, cd[q]);
                }
            }
        }
#else
        if (g.op1 != g.op0) flat_affine_k<K>(P.seg_affine[s], o, d, co, cd); // the chain as one affine map (composed at upload)
#endif
        flat_segment_k<K, MEDIA, HYBRID>(sc, P, g, s, o, d, co, cd, time, live, tmin, xi, best_t, best_hit, sub, tc);
    }
    }
}

#if !VK_STRICT
// trace_flat_k without media or subtrees, for a program of a shape compiled in (FlatShape, vk_internal.h): the same
// entries in the same order with the same arithmetic, but every loop unrolled over the shape's counts, so each operand
// is a constant-bank load at a constant offset -- no walk over FlatSeg's byte ranges, no loop counters or branches.
template <class G, int K>
VKD void flat_segment_static(const FlatProgram& P, const float3 (&co)[K], const float3 (&cd)[K], float tmin, float (&best_t)[K],
                             uint32_t (&best_hit)[K]) {
    float3 ci[K];
#pragma unroll
    for (int q = 0; q < K; ++q) ci[q] = rcp3(cd[q]);
#pragma unroll
    for (int i = G::x0; i < G::x1; ++i) flat_rect_k<K, 0, false>(P.rects[i], co, cd, ci, tmin, best_t, best_hit);
#pragma unroll
    for (int i = G::y0; i < G::y1; ++i) flat_rect_k<K, 1, false>(P.rects[i], co, cd, ci, tmin, best_t, best_hit);
#pragma unroll
    for (int i = G::z0; i < G::z1; ++i) flat_rect_k<K, 2, false>(P.rects[i], co, cd, ci, tmin, best_t, best_hit);
#pragma unroll
    for (int i = G::b0; i < G::b1; ++i) flat_box_k<K>(P.boxes[i], co, ci, tmin, best_t, best_hit);
#pragma unroll
    for (int i = G::s0; i < G::s1; ++i) flat_sphere_k<K>(P.spheres[i], co, cd, tmin, best_t, best_hit);
}
template <int K, int S, class G, class... Rest>
VKD void flat_segments_static(const FlatProgram& P, const float3 (&o)[K], const float3 (&d)[K], float tmin, float (&best_t)[K],
                              uint32_t (&best_hit)[K]) {
    if constexpr (S == 0) { // the world frame: the ray as it is
        flat_segment_static<G, K>(P, o, d, tmin, best_t, best_hit);
    } else {
        float3 co[K], cd[K];
        flat_affine_k<K>(P.seg_affine[S], o, d, co, cd);
        flat_segment_static<G, K>(P, co, cd, tmin, best_t, best_hit);
    }
    if constexpr (sizeof...(Rest) > 0) flat_segments_static<K, S + 1, Rest...>(P, o, d, tmin, best_t, best_hit);
}
template <int K, class... Seg>
VKD void trace_flat_static(const FlatProgram& P, FlatShape<Seg...>, const float3 (&o)[K], const float3 (&d)[K], float tmin, float (&best_t)[K],
                           uint32_t (&best_hit)[K]) {
#pragma unroll
    for (int q = 0; q < K; ++q) {
        best_t[q] = CUDART_INF_F;
        best_hit[q] = 0xFFFFFFFFu;
    }
    flat_segments_static<K, 0, Seg...>(P, o, d, tmin, best_t, best_hit);
}
#endif

// ---------------------------------------------------------------------------------------------
// HitRec (src/hittable.rs:11-31) of the winning primitive, built once per segment.
// ---------------------------------------------------------------------------------------------
struct HitRecD {
    float3 p, normal;
    float t, u, v;
    uint32_t front, mat;
    uint4 m; // materials[mat], fetched once per segment
};

// Out of line (atan2f + asinf are ~160 instructions and only image-textured spheres need them); by
// value, so that the caller's HitRec stays in registers.
static __device__ __noinline__ float2 spherical_uv(float px, float py, float pz) { // Sphere::spherical src/hittable.rs:54-61
    const float phi = atan2f(pz, px);
    const float theta = asinf(py);
    return make_float2(1.0f - ((phi + VK_PI) / (2.0f * VK_PI)), (theta + VK_PI / 2.0f) / VK_PI);
}
VKD void spherical(float3 p, float& u, float& v) {
    const float2 uv = spherical_uv(p.x, p.y, p.z);
    u = uv.x;
    v = uv.y;
}
VKD void set_face_normal(float3 dir, float3 outward, HitRecD& rec) { // src/hittable.rs:23-30
    rec.front = dot3(dir, outward) < 0.0f ? 1u : 0u;
    rec.normal = rec.front ? outward : -outward;
}
VKD void rect_record(float4 bounds, float k, uint32_t axes, uint32_t flip, float3 o, float3 d, float t, bool want_uv,
                     HitRecD& rec) { // src/hittable.rs:240-255 (+ FlipFace :300-308)
    (void)k;
    const uint32_t a0 = axes & 3u, a1 = (axes >> 2) & 3u, a2 = (axes >> 4) & 3u;
    rec.p = at(o, d, t);
    set_face_normal(d, f3(a2 == 0 ? 1.0f : 0.0f, a2 == 1 ? 1.0f : 0.0f, a2 == 2 ? 1.0f : 0.0f), rec);
    if (flip) rec.front ^= 1u;
    if (want_uv) {
        const float a = comp(o, a0) + t * comp(d, a0);
        const float b = comp(o, a1) + t * comp(d, a1);
        rec.u = (a - bounds.x) / (bounds.y - bounds.x);
        rec.v = (b - bounds.z) / (bounds.w - bounds.z);
    }
}
// the rect record of side `face` of a box (Boxy::new order)
VKD void box_side(float3 mn, float3 mx, uint32_t face, float4& bounds, float& k, uint32_t& axes) {
    switch (face >> 1) {
    case 0: bounds = make_float4(mn.x, mx.x, mn.y, mx.y); k = (face & 1u) ? mn.z : mx.z; axes = 0u | (1u << 2) | (2u << 4); break;
    case 1: bounds = make_float4(mn.x, mx.x, mn.z, mx.z); k = (face & 1u) ? mn.y : mx.y; axes = 0u | (2u << 2) | (1u << 4); break;
    default: bounds = make_float4(mn.y, mx.y, mn.z, mx.z); k = (face & 1u) ? mn.x : mx.x; axes = 1u | (2u << 2) | (0u << 4); break;
    }
}
// Full record of a leaf primitive hit at distance t by the ray (o, d) of the leaf's frame.
// (u, v) cost an atan2 + asin on a sphere: they are computed only when a texture of the hit
// material reads them (VKD_MAT_NEEDS_UV, set at upload) or the caller wants the full record.
VKD void leaf_record(const DScene& sc, uint32_t ref, uint32_t face, float3 o, float3 d, float time, float t, bool always_uv,
                     HitRecD& rec) {
    const uint32_t i = VKD_INDEX(ref);
    rec.t = t;
    rec.u = 0.0f;
    rec.v = 0.0f;
    bool want_uv = always_uv;
#if VK_SIMPLE
    want_uv = false; // no texture reads (u, v)
#endif
    switch (VKD_TYPE(ref)) {
    case VK_T_SPHERE:
#if !VK_SIMPLE
    case VK_T_MSPHERE:
#endif
    { // src/hittable.rs:76-89, :165-178
        float3 c;
        float radius;
        if (VK_SIMPLE || VKD_TYPE(ref) == VK_T_SPHERE) {
            const float4 s = __ldg(&sc.spheres[i]);
            c = f3(s);
            radius = s.w;
            rec.mat = __ldg(&sc.sphere_mat[i]);
        } else {
            const float4 m0 = __ldg(&sc.mspheres[3 * i]), m1 = __ldg(&sc.mspheres[3 * i + 1]), m2 = __ldg(&sc.mspheres[3 * i + 2]);
            c = msphere_center(m0, m1, m2.x, time);
            radius = m0.w;
            rec.mat = __float_as_uint(m2.y);
        }
        rec.m = __ldg(&sc.materials[rec.mat]);
        want_uv = !VK_SIMPLE && (want_uv || (rec.m.w & VKD_MAT_NEEDS_UV));
        rec.p = at(o, d, t);
        const float3 outward = (rec.p - c) / radius;
        set_face_normal(d, outward, rec);
        if (want_uv) spherical(outward, rec.u, rec.v);
        break;
    }
    case VK_T_RECT: {
        const float4 r0 = __ldg(&sc.rects[2 * i]), r1 = __ldg(&sc.rects[2 * i + 1]);
        const uint32_t axes = __float_as_uint(r1.y);
        rec.mat = __float_as_uint(r1.z);
        rec.m = __ldg(&sc.materials[rec.mat]);
        want_uv = !VK_SIMPLE && (want_uv || (rec.m.w & VKD_MAT_NEEDS_UV));
        rect_record(r0, r1.x, axes, axes & VK_RECT_FLIP, o, d, t, want_uv, rec);
        break;
    }
    case VK_T_BOX: {
        const float4 b0 = __ldg(&sc.boxes[2 * i]), b1 = __ldg(&sc.boxes[2 * i + 1]);
        float4 bounds;
        float k;
        uint32_t axes;
        box_side(f3(b0), f3(b1), face, bounds, k, axes);
        rec.mat = __float_as_uint(b0.w);
        rec.m = __ldg(&sc.materials[rec.mat]);
        want_uv = !VK_SIMPLE && (want_uv || (rec.m.w & VKD_MAT_NEEDS_UV));
        rect_record(bounds, k, axes, face & 1u, o, d, t, want_uv, rec);
        break;
    }
    default: break;
    }
}

// Build the HitRec the reference's `world.hit()` returns for the winning (prim, inst, t):
// re-walk the wrapper chain down (same operations -> same bits), make the leaf record in the
// object frame, then apply each wrapper's output stage on the way back up, including the
// set_face_normal calls with the child-frame ray (Translate :519, Rotate :618/:707/:796 -- Q9).
VKD void resolve_hit(const DScene& sc, const TraceHit& h, float3 o, float3 d, float time, bool always_uv, HitRecD& rec) {
    uint32_t kinds[VK_MAX_XFORM_DEPTH];
    float4 prm[VK_MAX_XFORM_DEPTH];
    float3 dchild[VK_MAX_XFORM_DEPTH];
    int nl = 0;
    float3 ro = o, rd = d;
    uint32_t ref = h.inst;
#pragma unroll 1
    while (VKD_TYPE(ref) == VK_T_XFORM && nl < VK_MAX_XFORM_DEPTH) {
        const float4 x0 = __ldg(&sc.xforms[2 * VKD_INDEX(ref)]);
        const float4 x1 = __ldg(&sc.xforms[2 * VKD_INDEX(ref) + 1]);
        const uint32_t kind = __float_as_uint(x0.x);
        if (kind == VK_X_TRANSLATE) ro = ro - f3(x1);
        else if (kind != VK_X_FLIP) {
            rot_fwd(kind, x1.x, x1.y, ro);
            rot_fwd(kind, x1.x, x1.y, rd);
        }
        kinds[nl] = kind;
        prm[nl] = x1;
        dchild[nl] = rd;
        ++nl;
        ref = __float_as_uint(x0.y);
    }
    if (VKD_TYPE(h.prim) == VK_T_MEDIUM) { // src/hittable.rs:481-489
        const float4 m = __ldg(&sc.media[VKD_INDEX(h.prim)]);
        rec.mat = __float_as_uint(m.z);
        rec.m = __ldg(&sc.materials[rec.mat]);
        rec.t = h.t;
        rec.p = at(ro, rd, h.t);
        rec.normal = f3(1.0f, 0.0f, 0.0f);
        rec.front = 1u;
        rec.u = 0.0f;
        rec.v = 0.0f;
        if (!VK_SIMPLE && (always_uv || (rec.m.w & VKD_MAT_NEEDS_UV))) { // (u, v) of rec1, the boundary entry hit
            float3 bo = ro, bd = rd;
            const uint32_t b = chain_down(sc, __float_as_uint(m.x), bo, bd);
            float t1;
            uint32_t face;
            if (leaf_t(sc, b, bo, bd, rcp3(bd), time, -CUDART_INF_F, CUDART_INF_F, t1, face)) {
                HitRecD r1;
                leaf_record(sc, b, face, bo, bd, time, t1, true, r1);
                rec.u = r1.u;
                rec.v = r1.v;
            }
        }
    } else {
        leaf_record(sc, h.prim, h.face, ro, rd, time, h.t, always_uv, rec);
    }
#pragma unroll 1
    for (int l = nl - 1; l >= 0; --l) {
        const uint32_t kind = kinds[l];
        if (kind == VK_X_FLIP) {
            rec.front ^= 1u;
        } else if (kind == VK_X_TRANSLATE) {
            rec.p = rec.p + f3(prm[l]);
            set_face_normal(dchild[l], rec.normal, rec);
        } else {
            rot_back(kind, prm[l].x, prm[l].y, rec.p);
            float3 n = rec.normal;
            rot_back(kind, prm[l].x, prm[l].y, n);
            set_face_normal(dchild[l], n, rec);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Textures (src/material.rs:228-434)
// ---------------------------------------------------------------------------------------------
VKD float perlin_noise(const float4* __restrict__ vec, const uint8_t* __restrict__ perm, float3 p) { // :392-413 + :331-352
    const float fx = floorf(p.x), fy = floorf(p.y), fz = floorf(p.z);
    const float u = p.x - fx, v = p.y - fy, w = p.z - fz;
    const uint32_t i = __float2uint_rz(fx), j = __float2uint_rz(fy), k = __float2uint_rz(fz); // saturating `as usize` (Q16)
    const float uu = u * u * (3.0f - 2.0f * u), vv = v * v * (3.0f - 2.0f * v), ww = w * w * (3.0f - 2.0f * w);
    float accum = 0.0f;
#pragma unroll
    for (uint32_t di = 0; di < 2; ++di)
#pragma unroll
        for (uint32_t dj = 0; dj < 2; ++dj)
#pragma unroll
            for (uint32_t dk = 0; dk < 2; ++dk) {
                const uint32_t idx = perm[(i + di) & 255u] ^ perm[256u + ((j + dj) & 255u)] ^ perm[512u + ((k + dk) & 255u)];
                const float4 c = __ldg(&vec[idx]);
                const float fi = (float)di, fj = (float)dj, fk = (float)dk;
                accum += (fi * uu + (1.0f - fi) * (1.0f - uu)) * (fj * vv + (1.0f - fj) * (1.0f - vv)) *
                         (fk * ww + (1.0f - fk) * (1.0f - ww)) * dot3(f3(c), f3(u - fi, v - fj, w - fk));
            }
    return accum;
}
VKD float perlin_turb(const float4* vec, const uint8_t* perm, float3 p, int depth) { // :379-390
    float accum = 0.0f, weight = 1.0f;
    float3 tp = p;
#pragma unroll 1
    for (int i = 0; i < depth; ++i) {
        accum += weight * perlin_noise(vec, perm, tp);
        weight *= 0.5f;
        tp = tp * 2.0f;
    }
    return fabsf(accum);
}
VKD float clamp_ref(float x, float mn, float mx) { return x < mn ? mn : (x > mx ? mx : x); } // Vec3::clamp keeps NaN
static __device__ __noinline__ float3 tex_value_general(const DScene& sc, uint4 t, float u, float v, float3 p);
VKD float3 tex_value(const DScene& sc, uint32_t ti, float u, float v, float3 p) {
    const uint4 t = __ldg(&sc.textures[ti]);
#if VK_SIMPLE
    (void)u, (void)v, (void)p;
    return f3(__uint_as_float(t.y), __uint_as_float(t.z), __uint_as_float(t.w)); // SolidColor :238-242 (the only kind)
#else
    if (t.x == VK_TEX_SOLID) return f3(__uint_as_float(t.y), __uint_as_float(t.z), __uint_as_float(t.w)); // SolidColor :238-242
    return tex_value_general(sc, t, u, v, p);
#endif
}
static __device__ __noinline__ float3 tex_value_general(const DScene& sc, uint4 t, float u, float v, float3 p) {
#pragma unroll 1
    for (int guard = 0; t.x == VK_TEX_CHECKER && guard < 16; ++guard) { // Checker :250-258 (sinf, not __sinf: args ~1e3)
        const float sins = sinf(10.0f * p.x) * sinf(10.0f * p.y) * sinf(10.0f * p.z);
        t = __ldg(&sc.textures[sins < 0.0f ? t.y : t.z]);
    }
    if (t.x == VK_TEX_SOLID) return f3(__uint_as_float(t.y), __uint_as_float(t.z), __uint_as_float(t.w));
    if (t.x == VK_TEX_IMAGE) { // ImageTexture::value :282-303, nearest texel, v flipped, RGB8
        const uint32_t width = t.z, height = t.w;
        const float uc = clamp_ref(u, 0.0f, 1.0f);
        const float vc = 1.0f - clamp_ref(v, 0.0f, 1.0f);
        uint32_t i = __float2uint_rz(uc * (float)width);
        uint32_t j = __float2uint_rz(vc * (float)height);
        if (i >= width) i = width - 1;
        if (j >= height) j = height - 1;
        const uint8_t* pix = sc.texels + (size_t)t.y + ((size_t)j * width + i) * 3u;
        const float s = 1.0f / 255.0f;
        return f3(s * (float)__ldg(pix), s * (float)__ldg(pix + 1), s * (float)__ldg(pix + 2));
    }
    // NoiseTexture::value :430-433
    const float scale = __uint_as_float(t.z);
    const float turb = perlin_turb(sc.perlin_vec + 256u * t.y, sc.perlin_perm + 768u * t.y, p, 7);
    const float g = 0.5f * (1.0f + sinf(scale * p.z + 10.0f * turb));
    return f3(g, g, g);
}

// ---------------------------------------------------------------------------------------------
// util.rs: reflect / refract / schlick (:14-29), ONB (:94-110), cosine direction (:52-63)
// ---------------------------------------------------------------------------------------------
VKD float3 reflect(float3 v, float3 n) { return v - n * dot3(v, n) * 2.0f; }
VKD float3 refract(float3 uv, float3 n, float etai_over_etat) {
    const float cos_theta = -dot3(uv, n);
    const float3 r_out_parallel = (uv + n * cos_theta) * etai_over_etat;
    const float3 r_out_perp = n * -sqrtf(1.0f - length2(r_out_parallel)); // no abs under the sqrt (Q7)
    return r_out_parallel + r_out_perp;
}
VKD float schlick(float cosine, float ref_idx) {
    float r0 = (1.0f - ref_idx) / (1.0f + ref_idx);
    r0 = r0 * r0;
    const float x = 1.0f - cosine, x2 = x * x;
    return r0 + (1.0f - r0) * (x2 * x2 * x); // powf(5.0)
}
struct Onb {
    float3 u, v, w;
};
VKD Onb onb_from_w(float3 n) {
    Onb o;
    o.w = unit_vector(n);
    const float3 a = fabsf(o.w.x) > 0.9f ? f3(0.0f, 1.0f, 0.0f) : f3(1.0f, 0.0f, 0.0f);
    o.v = unit_vector(cross3(o.w, a));
    o.u = cross3(o.w, o.v);
    return o;
}
VKD float3 random_cosine_direction(float r1, float r2) {
    const float z = sqrtf(1.0f - r2);
    float s, c;
#if VK_STRICT
    sincosf(2.0f * r1 * VK_PI, &s, &c);
#else
    __sincosf(2.0f * r1 * VK_PI, &s, &c);
#endif
    const float sr = sqrtf(r2);
    return f3(c * sr, s * sr, z);
}
// random_in_unit_sphere (:31-39) without the rejection loop: uniform direction x cbrt(u) radius
// is the same distribution (uniform in the unit ball).
VKD float3 random_in_unit_sphere(float u1, float u2, float u3) {
    const float z = 1.0f - 2.0f * u1;
    const float r = sqrtf(fmaxf(0.0f, 1.0f - z * z));
    float s, c;
    __sincosf(2.0f * VK_PI * u2, &s, &c);
    const float rad = cbrtf(u3);
    return f3(r * c, r * s, z) * rad;
}

// ---------------------------------------------------------------------------------------------
// Light sampling: `impl Hittable for Vec<Arc<HittableSS>>` pdf_value / random
// (src/hittable.rs:420-433) over SceneConfig.lights, with the per-type implementations:
// Rect (:271-291), Sphere (:104-134, keeps the (1-z*z) bug Q18), Boxy (:371-377, whose flipped
// sides fall back to the trait defaults 0.0 / (1,0,0) :36-41).
// ---------------------------------------------------------------------------------------------
VKD float rect_pdf_value(float4 bounds, float k, uint32_t axes, float3 origin, float3 v) {
    float t;
    if (!rect_t(bounds, k, axes, origin, v, rcp3(v), 0.001f, CUDART_INF_F, t)) return 0.0f;
    const float area = (bounds.y - bounds.x) * (bounds.w - bounds.z);
    const float distance_squared = t * t * length2(v);
    // rec.normal is +-e_axis2, so |v . n| = |v[axis2]|
    const float cosine = fabsf(comp(v, (axes >> 4) & 3u)) / sqrtf(length2(v));
    return distance_squared / (cosine * area);
}
VKD float3 rect_random(float4 bounds, float k, uint32_t axes, float3 origin, uint32_t x0, uint32_t x1) {
    const uint32_t a0 = axes & 3u, a1 = (axes >> 2) & 3u;
    const float pa = gen_range(x0, bounds.x, bounds.y), pb = gen_range(x1, bounds.z, bounds.w);
    float3 pt;
    pt.x = a0 == 0 ? pa : (a1 == 0 ? pb : k);
    pt.y = a0 == 1 ? pa : (a1 == 1 ? pb : k);
    pt.z = a0 == 2 ? pa : (a1 == 2 ? pb : k);
    return pt - origin;
}
// The light list of every shipped scene holds one Rect; Sphere and Boxy lights are kept out of line so
// that the hot shading code stays small (the kernels are instruction-fetch sensitive, see DESIGN.md).
#if !VK_SIMPLE
static __device__ __noinline__ float light_pdf_value_other(const DScene& sc, uint32_t ref, float3 o, float3 v) {
    const uint32_t i = VKD_INDEX(ref);
    switch (VKD_TYPE(ref)) {
    case VK_T_SPHERE: {
        const float4 s = __ldg(&sc.spheres[i]);
        float t;
        if (!sphere_t(f3(s), s.w, o, v, 0.001f, CUDART_INF_F, t)) return 0.0f;
        const float cos_theta_max = sqrtf(1.0f - s.w * s.w / length2(f3(s) - o));
        const float solid_angle = 2.0f * VK_PI * (1.0f - cos_theta_max);
        return 1.0f / solid_angle;
    }
    case VK_T_BOX: {
        const float4 b0 = __ldg(&sc.boxes[2 * i]), b1 = __ldg(&sc.boxes[2 * i + 1]);
        const float weight = 1.0f / 6.0f;
        float sum = 0.0f;
#pragma unroll 1
        for (uint32_t f = 0; f < 6; ++f) {
            float4 bounds;
            float k;
            uint32_t axes;
            box_side(f3(b0), f3(b1), f, bounds, k, axes);
            sum += weight * ((f & 1u) ? 0.0f : rect_pdf_value(bounds, k, axes, o, v));
        }
        return sum;
    }
    default: return 0.0f; // Hittable::pdf_value default
    }
}
#endif
VKD float light_pdf_value(const DScene& sc, uint32_t ref, float3 o, float3 v) {
    if (VKD_TYPE(ref) == VK_T_RECT) {
        const uint32_t i = VKD_INDEX(ref);
        const float4 r0 = __ldg(&sc.rects[2 * i]), r1 = __ldg(&sc.rects[2 * i + 1]);
        if (__float_as_uint(r1.y) & VK_RECT_FLIP) return 0.0f; // FlipFace: trait default
        return rect_pdf_value(r0, r1.x, __float_as_uint(r1.y), o, v);
    }
#if VK_SIMPLE
    return 0.0f;
#else
    return light_pdf_value_other(sc, ref, o, v);
#endif
}
#if !VK_SIMPLE
static __device__ __noinline__ float3 light_random_other(const DScene& sc, uint32_t ref, float3 o, uint32_t x0, uint32_t x1, uint32_t x2) {
    const uint32_t i = VKD_INDEX(ref);
    switch (VKD_TYPE(ref)) {
    case VK_T_SPHERE: {
        const float4 s = __ldg(&sc.spheres[i]);
        const float3 direction = f3(s) - o;
        const float distance_squared = length2(direction);
        const Onb uvw = onb_from_w(direction);
        const float r1 = u01(x0), r2 = u01(x1);
        const float z = 1.0f + r2 * (sqrtf(1.0f - s.w * s.w / distance_squared) - 1.0f);
        float sn, cs;
        sincosf(2.0f * VK_PI * r1, &sn, &cs);
        const float x = cs * (1.0f - z * z), y = sn * (1.0f - z * z);
        return uvw.u * x + uvw.v * y + uvw.w * z;
    }
    case VK_T_BOX: {
        const float4 b0 = __ldg(&sc.boxes[2 * i]), b1 = __ldg(&sc.boxes[2 * i + 1]);
        const uint32_t f = min(5u, (uint32_t)(u01(x2) * 6.0f));
        if (f & 1u) return f3(1.0f, 0.0f, 0.0f);
        float4 bounds;
        float k;
        uint32_t axes;
        box_side(f3(b0), f3(b1), f, bounds, k, axes);
        return rect_random(bounds, k, axes, o, x0, x1);
    }
    default: return f3(1.0f, 0.0f, 0.0f); // Hittable::random default
    }
}
#endif
VKD float3 light_random(const DScene& sc, uint32_t ref, float3 o, uint32_t x0, uint32_t x1, uint32_t x2) {
    if (VKD_TYPE(ref) == VK_T_RECT) {
        const uint32_t i = VKD_INDEX(ref);
        const float4 r0 = __ldg(&sc.rects[2 * i]), r1 = __ldg(&sc.rects[2 * i + 1]);
        if (__float_as_uint(r1.y) & VK_RECT_FLIP) return f3(1.0f, 0.0f, 0.0f);
        return rect_random(r0, r1.x, __float_as_uint(r1.y), o, x0, x1);
    }
#if VK_SIMPLE
    (void)x2;
    return f3(1.0f, 0.0f, 0.0f);
#else
    return light_random_other(sc, ref, o, x0, x1, x2);
#endif
}
VKD float lights_pdf_value(const DScene& sc, float3 o, float3 v) {
#if VK_SIMPLE || VK_LIGHT0
    // (the one unflipped Rect light, from the kernel parameters: DScene::light0_a)
    return 0.0f + 1.0f * rect_pdf_value(sc.light0_a, sc.light0_b.x, __float_as_uint(sc.light0_b.y), o, v); // sum = 0.0 + weight * pdf with weight 1/1
#endif
    const float weight = 1.0f / (float)sc.n_lights;
    float sum = 0.0f;
#pragma unroll 1
    for (uint32_t l = 0; l < sc.n_lights; ++l) sum += weight * light_pdf_value(sc, __ldg(&sc.lights[l]), o, v);
    return sum;
}

// ---------------------------------------------------------------------------------------------
// The integrator's two per-sample pieces, shared by the megakernel (vk_kernels.cu) and the
// wavefront kernels (vk_wavefront.cu): camera ray generation and one bounce of ray_color.
// ---------------------------------------------------------------------------------------------
// Camera::get_ray (src/main.rs:111-120).  random_in_unit_disk() is always drawn by the reference
// and multiplied by lens_radius; with lens_radius == 0 the product is exactly 0, so the draw is
// skipped.  The disk sample is direct (sqrt-radius) instead of the rejection loop: same law.
// lens_radius * random_in_unit_disk() (src/main.rs:112-113), direct sampling instead of the rejection loop
static __device__ __noinline__ float2 camera_lens_disk(uint32_t pixel, uint32_t sample, uint32_t k0, uint32_t k1, float lens_radius) {
    const uint4 q = philox4x32_10(make_uint4(pixel, sample, 1u, 0u), make_uint2(k0, k1)); // block(depth 0, 1)
    const float rad = sqrtf(u01(q.x)) * lens_radius;
    float sn, cs;
    __sincosf(2.0f * VK_PI * u01(q.y), &sn, &cs);
    return make_float2(rad * cs, rad * sn);
}
VKD void camera_get_ray(const DCamera& cam, const PathRng& rng, uint32_t x, uint32_t y, uint32_t width, uint32_t height,
                        float3& o, float3& d, float& time) {
    const uint4 r = rng.block(0u, 0u);
    const float s = ((float)x + u01(r.x)) / (float)(width - 1);  // src/main.rs:187
    const float t = ((float)y + u01(r.y)) / (float)(height - 1); // src/main.rs:188
    float3 offset = f3(0.0f, 0.0f, 0.0f);
    if (cam.lens_radius != 0.0f) { // no shipped scene has an aperture: out of line, everything by value
        const float2 disk = camera_lens_disk(rng.pixel, rng.sample, rng.key.x, rng.key.y, cam.lens_radius);
        offset = cam.u * disk.x + cam.v * disk.y;
    }
    o = cam.origin + offset;
    d = cam.lower_left_corner + cam.horizontal * s + cam.vertical * t - cam.origin - offset;
    time = gen_range(r.z, cam.time0, cam.time1);
}

// Where a bounce takes its variates from: the path's Philox stream (block 0 of the segment; block 9 for
// SpecDiffuse's choice), or a table the caller supplies (vk_eval, the per-function parity hook).
struct BounceXiPhilox {
    const PathRng& rng;
    uint32_t depth;
    VKD uint4 block0() const { return rng.block(depth, 0u); }
    VKD uint32_t spec() const { return rng.block(depth, 9u).x; }
};
struct BounceXiTable {
    uint4 r;
    uint32_t s;
    VKD uint4 block0() const { return r; }
    VKD uint32_t spec() const { return s; }
};
// One bounce of ray_color's loop body after world.hit() returned `rec` (src/main.rs:131-149), one body per material
// class: shade_xi dispatches on the material; a warp-queue shade batch whose queue fixes the class calls its body
// directly (wq_shade_batch), so that it carries no code of the other classes.
// DiffuseLight (src/material.rs:218-225; scatter_with_pdf -> None; src/main.rs:147-149): the path ends.
VKD bool shade_emitter(const DScene& sc, const HitRecD& rec, const uint4& m, const float3& beta, float3& L) {
    float3 emitted = f3(0.0f, 0.0f, 0.0f);
    if (rec.front) emitted = tex_value(sc, m.y, rec.u, rec.v, rec.p);
    L = L + beta * emitted;
    return false;
}
// Dielectric (src/material.rs:177-206), attenuation (1,1,1).
VKD bool shade_dielectric(const HitRecD& rec, const uint4& m, const uint4& r, float3& o, float3& d) {
    const float ref_idx = __uint_as_float(m.z);
    const float etai_over_etat = rec.front ? 1.0f / ref_idx : ref_idx;
    const float3 unit_direction = unit_vector(d);
    const float cos_theta = fminf(dot3(-unit_direction, rec.normal), 1.0f);
    const float sin_theta = sqrtf(1.0f - cos_theta * cos_theta);
    float3 nd;
    if (etai_over_etat * sin_theta > 1.0f) nd = reflect(unit_direction, rec.normal);
    else if (u01(r.x) < schlick(cos_theta, etai_over_etat)) nd = reflect(unit_direction, rec.normal);
    else nd = refract(unit_direction, rec.normal, etai_over_etat);
    o = rec.p;
    d = nd; // keeps r.time
    return true;
}
// Lambertian / Isotropic (src/material.rs:92-108, :448-464): cosine lobe about rec.normal,
// mixed 50/50 with light sampling (src/main.rs:139-146).  spdf_type: whose scattering_pdf applies.
VKD bool shade_diffuse(const DScene& sc, const HitRecD& rec, const uint4& m, uint32_t spdf_type, const uint4& r, float3& o, float3& d,
                       float3& beta, bool& valid) {
    const float3 attenuation = tex_value(sc, m.y, rec.u, rec.v, rec.p);
#if VK_STRICT
    const Onb uvw = onb_from_w(rec.normal);
    const float3 onb_w = uvw.w;
#else
    const float3 onb_w = unit_vector(rec.normal); // ONB::new_from_w: w; u and v are built only where they are used
#endif
    float3 nd;
    if (u01(r.x) < 0.5f) { // MixturePDF::generate src/util.rs:177-185 -> HittablePDF -> list random
#if VK_SIMPLE || VK_LIGHT0
        nd = rect_random(sc.light0_a, sc.light0_b.x, __float_as_uint(sc.light0_b.y), rec.p, r.y, r.z); // the one (unflipped Rect) light
#else
        const uint32_t li = sc.n_lights > 1 ? min(sc.n_lights - 1u, (uint32_t)(u01(r.w) * (float)sc.n_lights)) : 0u;
        nd = light_random(sc, __ldg(&sc.lights[li]), rec.p, r.y, r.z, r.w * 0x9E3779B1u);
#endif
    } else {
        const float3 c = random_cosine_direction(u01(r.y), u01(r.z));
#if !VK_STRICT
        const Onb uvw = onb_from_w(rec.normal);
#endif
        nd = uvw.u * c.x + uvw.v * c.y + uvw.w * c.z;
    }
    const float3 und = unit_vector(nd);
    const float cos_w = dot3(und, onb_w);
    const float cosine_pdf = cos_w <= 0.0f ? 0.0f : cos_w / VK_PI;                // CosinePDF::value src/util.rs:134-142
    const float pdf = 0.5f * lights_pdf_value(sc, rec.p, nd) + 0.5f * cosine_pdf; // MixturePDF::value :173-175
    float spdf = 0.0f;                                                            // Material::scattering_pdf default
    if (spdf_type == VK_M_LAMBERTIAN || spdf_type == VK_M_ISOTROPIC) {
        const float cos_n = dot3(rec.normal, und);
        spdf = cos_n < 0.0f ? 0.0f : cos_n / VK_PI;
    }
#if VK_STRICT
    const float3 w = f3(attenuation.x * spdf / pdf, attenuation.y * spdf / pdf, attenuation.z * spdf / pdf);
#else
    const float3 w = attenuation * (spdf / pdf); // one division (same value up to rounding; 0 / 0 and x / 0 stay NaN / inf)
#endif
    if (!finite3(w)) { // reference: NaN/Inf poisons the sample, which main.rs:192 then drops (Q3)
        valid = false;
        return false;
    }
    beta = beta * w;
    if (beta.x == 0.0f && beta.y == 0.0f && beta.z == 0.0f) return false; // nothing further can contribute
    o = rec.p;
    d = nd; // Ray::new_with_time(c.p, dir, r.time): keeps the camera-sampled time
    return true;
}
// Returns false when the path ends.  `valid` is cleared when the reference's value would be
// non-finite (the whole sample is then dropped, src/main.rs:191-194).
template <class XI>
VKD bool shade_xi(const DScene& sc, const HitRecD& rec, const XI& xi, float3& o, float3& d, float& time,
                  float3& beta, float3& L, bool& valid) {
    uint4 m = rec.m;
    uint32_t type = m.x;
    uint32_t spdf_type = type; // whose scattering_pdf applies
    if (!VK_SIMPLE && !VK_LIGHT0 && type == VK_M_SPECDIFFUSE) { // src/material.rs:474-488: emitted() is the trait default (0)
        const uint32_t diffuse = m.w & ~VKD_MAT_NEEDS_UV;
        spdf_type = __ldg(&sc.materials[diffuse]).x;
        m = __ldg(&sc.materials[u01(xi.spec()) < __uint_as_float(m.z) ? m.y : diffuse]);
        type = m.x;
        if (type == VK_M_DIFFUSE_LIGHT) { // emitted() of the SpecDiffuse is 0 (src/main.rs:147-149)
            L = L + beta * f3(0.0f, 0.0f, 0.0f);
            return false;
        }
    } else if (type == VK_M_DIFFUSE_LIGHT) {
        return shade_emitter(sc, rec, m, beta, L);
    }
    const uint4 r = xi.block0();
    if (type == VK_M_DIELECTRIC) return shade_dielectric(rec, m, r, o, d);
    if (!VK_SIMPLE && type == VK_M_METAL) { // src/material.rs:134-141: Ray::new -> time 0 (Q6), never absorbed
        const float fuzz = __uint_as_float(m.z);
        float3 nd = reflect(unit_vector(d), rec.normal);
        if (fuzz != 0.0f) nd = nd + random_in_unit_sphere(u01(r.x), u01(r.y), u01(r.z)) * fuzz;
        beta = beta * tex_value(sc, m.y, rec.u, rec.v, rec.p);
        o = rec.p;
        d = nd;
        time = 0.0f;
        return true;
    }
    return shade_diffuse(sc, rec, m, spdf_type, r, o, d, beta, valid);
}
VKD bool shade(const DScene& sc, const HitRecD& rec, const PathRng& rng, uint32_t depth, float3& o, float3& d, float& time,
               float3& beta, float3& L, bool& valid) {
    const BounceXiPhilox xi = {rng, depth};
    return shade_xi(sc, rec, xi, o, d, time, beta, L, valid);
}

// Sample end (src/main.rs:191-194, `c += color` for a finite sample): three integer atomics into the pixel's
// fixed-point sums (see RenderBuffers), which makes the frame independent of who adds what when.  A zero
// component adds nothing and is skipped (most paths end on weight 0 or on a black miss).
VKD void accumulate_sample(const RenderBuffers& buf, uint32_t pixel, float3 L) {
    unsigned long long* p = buf.acc + (size_t)pixel * 3u;
    const float lim = 4294967296.0f; // 2^32 * 2^30 fits the 64-bit accumulator
    if (L.x != 0.0f) atomicAdd(p + 0, (unsigned long long)__float2ll_rn(fminf(fmaxf(L.x, -lim), lim) * VK_ACC_SCALE));
    if (L.y != 0.0f) atomicAdd(p + 1, (unsigned long long)__float2ll_rn(fminf(fmaxf(L.y, -lim), lim) * VK_ACC_SCALE));
    if (L.z != 0.0f) atomicAdd(p + 2, (unsigned long long)__float2ll_rn(fminf(fmaxf(L.z, -lim), lim) * VK_ACC_SCALE));
    if (buf.accsq) {
        double* q = buf.accsq + (size_t)pixel * 3u;
        if (L.x != 0.0f) atomicAdd(q + 0, (double)L.x * (double)L.x);
        if (L.y != 0.0f) atomicAdd(q + 1, (double)L.y * (double)L.y);
        if (L.z != 0.0f) atomicAdd(q + 2, (double)L.z * (double)L.z);
    }
}
// The list kernels of an adaptive pass (ListArgs) add, next to accumulate_sample, each channel's square to the pixel's
// fixed-point sums of squares: |L| clamped to VK_SQ_CLAMP, squared exactly in double (a float product fits its mantissa),
// rounded to VK_SQ_SCALE units.  Integer sums again, so the stopping statistic does not depend on arrival order.
VKD void accumulate_square(unsigned long long* sq, uint32_t pixel, float3 L) {
    unsigned long long* q = sq + (size_t)pixel * 3u;
    const double cx = fminf(fabsf(L.x), VK_SQ_CLAMP), cy = fminf(fabsf(L.y), VK_SQ_CLAMP), cz = fminf(fabsf(L.z), VK_SQ_CLAMP);
    if (L.x != 0.0f) atomicAdd(q + 0, __double2ull_rn(cx * cx * (double)VK_SQ_SCALE));
    if (L.y != 0.0f) atomicAdd(q + 1, __double2ull_rn(cy * cy * (double)VK_SQ_SCALE));
    if (L.z != 0.0f) atomicAdd(q + 2, __double2ull_rn(cz * cz * (double)VK_SQ_SCALE));
}

// ---------------------------------------------------------------------------------------------
// Work domains (OneFrame, FrameArgs, ListArgs: vk_internal.h): what a render kernel's body asks its domain (the warp
// queues' chunk dealing is next to WqCtx, vk_warpq.cuh).  Each question has a one-frame answer as its template and
// an overload for each domain that answers differently; for OneFrame every answer is the single-frame code itself or
// a constant that folds away.
// ---------------------------------------------------------------------------------------------
// Philox key of frame f of a batch: seed + f, the key vecchio_gpu_render --seed gives frame f of a frame loop
VKD uint2 frame_key(const RenderArgs& a, uint32_t f) {
    const unsigned long long k = (((unsigned long long)a.seed_hi << 32) | a.seed_lo) + f;
    return make_uint2((uint32_t)k, (uint32_t)(k >> 32));
}
// the domain's unit count as a multiple of one frame's
template <class D> VKD uint32_t dom_frames(const D&) { return 1u; }
VKD uint32_t dom_frames(const FrameArgs& fr) { return fr.n_frames; }
// the pixels a frame's units run over: W*H, or the list (a unit's "pixel" is then a list index, see dom_list_pixel)
template <class D> VKD uint32_t dom_pixels(const D&, const RenderArgs& a) { return a.width * a.height; }
VKD uint32_t dom_pixels(const ListArgs& ls, const RenderArgs&) { return ls.n; }
VKD uint32_t dom_pixels(const FrameListArgs& fl, const RenderArgs&) { return fl.ls.n; }
template <class D> VKD uint32_t dom_list_pixel(const D&, uint32_t i) { return i; }
VKD uint32_t dom_list_pixel(const ListArgs& ls, uint32_t i) { return ls.list[i]; }
VKD uint32_t dom_list_pixel(const FrameListArgs& fl, uint32_t i) { return fl.ls.list[i]; } // (batch-wide: see dom_unit_frame)
// Frame-major units: u of `per` units per frame -> its frame, and u within that frame (one frame: 0, u unchanged)
template <class D, class T> VKD uint32_t dom_split_frame(const D&, T&, T) { return 0u; }
template <class T> VKD uint32_t dom_split_frame(const FrameArgs&, T& u, T per) {
    const uint32_t f = (uint32_t)(u / per);
    u -= (T)f * per;
    return f;
}
// frame f's first accumulator pixel, camera and Philox key (rng.key arrives as the seed's)
template <class D> VKD uint32_t dom_plane(const D&, uint32_t) { return 0u; }
VKD uint32_t dom_plane(const FrameArgs& fr, uint32_t f) { return f * fr.n_pix; }
template <class D> VKD const DCamera& dom_camera(const D&, const DCamera& cam, uint32_t) { return cam; }
VKD const DCamera& dom_camera(const FrameArgs& fr, const DCamera&, uint32_t f) { return fr.cams[f]; }
VKD const DCamera& dom_camera(const FrameListArgs& fl, const DCamera&, uint32_t f) { return fl.fr.cams[f]; }
template <class D> VKD void dom_frame_key(const D&, const RenderArgs&, uint32_t, PathRng&) {}
VKD void dom_frame_key(const FrameArgs&, const RenderArgs& a, uint32_t f, PathRng& rng) { rng.key = frame_key(a, f); }
// The pixel a warp-queue slot keeps (rng.pixel, the accumulator index: batch-wide in a batch) -> the Philox counter's
// pixel and key of its frame
template <class D> VKD void dom_slot_rng(const D&, const RenderArgs&, PathRng&) {}
VKD void dom_slot_rng(const FrameArgs& fr, const RenderArgs& a, PathRng& rng) {
    const uint32_t f = rng.pixel / fr.n_pix;
    rng.pixel = rng.pixel - f * fr.n_pix;
    rng.key = frame_key(a, f);
}
VKD void dom_slot_rng(const FrameListArgs& fl, const RenderArgs& a, PathRng& rng) { dom_slot_rng(fl.fr, a, rng); }
// Only a list across frames has a frame per unit rather than per item (the lane megakernels ask this when a unit's
// rng.pixel holds its list entry, the batch-wide pixel): rng.pixel becomes the frame's pixel, rng.key the frame's key, and
// the frame is returned.  Its accumulator pixel is then plane + rng.pixel, its camera dom_camera(dom, cam, f).
template <class D> struct dom_frame_per_unit { static constexpr bool value = false; };
template <> struct dom_frame_per_unit<FrameListArgs> { static constexpr bool value = true; };
VKD uint32_t dom_unit_frame(const FrameListArgs& fl, const RenderArgs& a, PathRng& rng) {
    const uint32_t f = rng.pixel / fl.fr.n_pix;
    dom_slot_rng(fl.fr, a, rng);
    return f;
}
// a finished, finite sample into accumulator pixel `pixel`; an adaptive pass also keeps its squares
template <class D> VKD void dom_accumulate(const D&, const RenderBuffers& buf, uint32_t pixel, float3 L) { accumulate_sample(buf, pixel, L); }
VKD void dom_accumulate(const ListArgs& ls, const RenderBuffers& buf, uint32_t pixel, float3 L) {
    accumulate_sample(buf, pixel, L);
    accumulate_square(ls.sq, pixel, L);
}
VKD void dom_accumulate(const FrameListArgs& fl, const RenderBuffers& buf, uint32_t pixel, float3 L) { dom_accumulate(fl.ls, buf, pixel, L); }
// Unit u of a lane-megakernel item: pixel (px0, py0) + (u & 7, u >> 3 & 3) of an 8x4 tile -> (px, py) and the frame pixel
// index; false for a unit outside the image.  A list's "tile" is 32 consecutive entries, unit u takes entry u & 31.
template <class D>
VKD bool mk_unit(const D&, const RenderArgs& a, uint32_t, uint32_t px0, uint32_t py0, uint32_t u, uint32_t& px, uint32_t& py, uint32_t& pixel) {
    px = px0 + (u & 7u);
    py = py0 + ((u >> 3) & 3u);
    if (!(px < a.width && py < a.height)) return false; // ragged tiles: a unit outside the image is void
    pixel = py * a.width + px;                          // i = y*width + x, row 0 = bottom (src/main.rs:182-183)
    return true;
}
VKD bool mk_unit(const ListArgs& ls, const RenderArgs& a, uint32_t tile, uint32_t, uint32_t, uint32_t u, uint32_t& px, uint32_t& py,
                 uint32_t& pixel) {
    const uint32_t li = tile * 32u + (u & 31u);
    if (!(li < ls.n)) return false; // the last group of the list is ragged
    pixel = ls.list[li];
    py = pixel / a.width;
    px = pixel - py * a.width;
    return true;
}
// over a list across frames `pixel` is the batch-wide entry (the body resolves its frame with dom_unit_frame), (px, py) its frame's
VKD bool mk_unit(const FrameListArgs& fl, const RenderArgs& a, uint32_t tile, uint32_t, uint32_t, uint32_t u, uint32_t& px, uint32_t& py,
                 uint32_t& pixel) {
    const uint32_t li = tile * 32u + (u & 31u);
    if (!(li < fl.ls.n)) return false;
    pixel = fl.ls.list[li];
    const uint32_t p = pixel % fl.fr.n_pix;
    py = p / a.width;
    px = p - py * a.width;
    return true;
}

// A ray that leaves the scene: the constant background of src/main.rs:124,151, or with
// VK_FLAG_SKY_BACKGROUND the book-1 sky (1-t)*white + t*(0.5,0.7,1.0), t = 0.5*(unit(d).y + 1).
VKD float3 miss_color(const RenderArgs& a, float3 d) {
    if (!(a.flags & VK_FLAG_SKY_BACKGROUND)) return a.background;
    const float t = 0.5f * (unit_vector(d).y + 1.0f);
    return f3(1.0f, 1.0f, 1.0f) * (1.0f - t) + f3(0.5f, 0.7f, 1.0f) * t;
}

// One bounce of the book-1/2 integrator built on the legacy `Material::scatter` methods
// (VK_FLAG_LEGACY_SCATTER): emitted + attenuation * ray_color(scattered), no light list, no PDFs.
// Lambertian src/material.rs:85-90 (+ :51-58), Metal :118-132, Dielectric :150-175,
// DiffuseLight :215-217, Isotropic :442-446.  SpecDiffuse has no legacy method of its own (its
// default `scatter` unwraps a missing specular ray and panics, :21-28): refused before the launch.
template <class XI>
VKD bool shade_legacy_xi(const DScene& sc, const HitRecD& rec, const XI& xi, float3& o, float3& d, float& time,
                         float3& beta, float3& L, bool& valid) {
    const uint4 m = rec.m;
    const uint32_t type = m.x;
    if (type == VK_M_DIFFUSE_LIGHT) { // scatter -> None: the path ends with the emission (if lit from the front)
        if (rec.front) L = L + beta * tex_value(sc, m.y, rec.u, rec.v, rec.p);
        return false;
    }
    if (type == VK_M_SPECDIFFUSE) {
        valid = false;
        return false;
    }
    const uint4 r = xi.block0();
    float3 nd;
    if (type == VK_M_DIELECTRIC) { // same body as scatter_with_pdf, attenuation (1,1,1), keeps r.time
        const float ref_idx = __uint_as_float(m.z);
        const float etai_over_etat = rec.front ? 1.0f / ref_idx : ref_idx;
        const float3 unit_direction = unit_vector(d);
        const float cos_theta = fminf(dot3(-unit_direction, rec.normal), 1.0f);
        const float sin_theta = sqrtf(1.0f - cos_theta * cos_theta);
        if (etai_over_etat * sin_theta > 1.0f) nd = reflect(unit_direction, rec.normal);
        else if (u01(r.x) < schlick(cos_theta, etai_over_etat)) nd = reflect(unit_direction, rec.normal);
        else nd = refract(unit_direction, rec.normal, etai_over_etat);
    } else if (type == VK_M_METAL) { // keeps r.time (unlike scatter_with_pdf); absorbed below the surface
        const float fuzz = __uint_as_float(m.z);
        nd = reflect(unit_vector(d), rec.normal);
        if (fuzz != 0.0f) nd = nd + random_in_unit_sphere(u01(r.x), u01(r.y), u01(r.z)) * fuzz;
        if (!(dot3(nd, rec.normal) > 0.0f)) return false; // None: emitted (0) is all that is left
        beta = beta * tex_value(sc, m.y, rec.u, rec.v, rec.p);
    } else if (type == VK_M_ISOTROPIC) {
        nd = random_in_unit_sphere(u01(r.x), u01(r.y), u01(r.z));
        beta = beta * tex_value(sc, m.y, rec.u, rec.v, rec.p);
    } else { // Lambertian: rec.normal + a uniform point on the unit sphere
        const float ang = gen_range(r.x, 0.0f, 2.0f * VK_PI), z = gen_range(r.y, -1.0f, 1.0f);
        const float rr = sqrtf(1.0f - z * z);
        float sn, cs;
        sincosf(ang, &sn, &cs);
        nd = rec.normal + f3(rr * cs, rr * sn, z);
        beta = beta * tex_value(sc, m.y, rec.u, rec.v, rec.p);
    }
    o = rec.p;
    d = nd;
    (void)time;
    return true;
}
VKD bool shade_legacy(const DScene& sc, const HitRecD& rec, const PathRng& rng, uint32_t depth, float3& o, float3& d, float& time,
                      float3& beta, float3& L, bool& valid) {
    const BounceXiPhilox xi = {rng, depth};
    return shade_legacy_xi(sc, rec, xi, o, d, time, beta, L, valid);
}

} // namespace VK_NS
