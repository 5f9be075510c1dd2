// vk_relayout.h -- host-side planning of the device layout of a flattened scene: validation, the 4-wide
// BVH collapse, the flat traversal program and the "simple scene" test.  Pure host code (no CUDA
// calls): vk_scene_upload copies what Relayout produces, vk_scene_check reports it without a device.
#pragma once
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "vk_internal.h"

namespace vkhost {

// ------------------------------------------------------------------------------------------------
// scene validation: everything the kernels assume is checked here, and anything the GPU path does
// not implement is refused with VK_ERR_UNSUPPORTED instead of being rendered wrongly.
// ------------------------------------------------------------------------------------------------
inline uint32_t __float_as_uint_host(float f) {
    uint32_t u;
    std::memcpy(&u, &f, 4);
    return u;
}
inline float __uint_as_float_host(uint32_t u) {
    float f;
    std::memcpy(&f, &u, 4);
    return f;
}
struct Validator {
    const vk_scene_desc* d;
    std::string err;
    int code = VK_OK;
    std::vector<int> node_depth;       // 0 = unvisited
    std::vector<uint8_t> node_medium;  // subtree holds a ConstantMedium
    std::vector<uint8_t> node_inchain; // visited below an instance
    std::vector<uint8_t> node_xform;   // subtree holds a transform (an instance, or a medium with a transformed boundary)
    int level = 0;                     // recursion depth of visit() (host stack guard)

    bool bad(int c, const std::string& m) {
        if (code == VK_OK) {
            code = c;
            err = m;
        }
        return false;
    }
    bool leaf_ok(vk_ref r) {
        const uint32_t i = VK_REF_INDEX(r);
        switch (VK_REF_TYPE(r)) {
        case VK_T_SPHERE: return i < d->n_spheres || bad(VK_ERR_INVALID, "sphere index out of range");
        case VK_T_MSPHERE: return i < d->n_mspheres || bad(VK_ERR_INVALID, "moving-sphere index out of range");
        case VK_T_RECT: return i < d->n_rects || bad(VK_ERR_INVALID, "rect index out of range");
        case VK_T_BOX: return i < d->n_boxes || bad(VK_ERR_INVALID, "box index out of range");
        default: return false;
        }
    }
    static bool is_leaf_type(uint32_t t) { return t == VK_T_SPHERE || t == VK_T_MSPHERE || t == VK_T_RECT || t == VK_T_BOX; }

    // returns the first non-wrapper ref of a chain starting at r (or NONE on error)
    vk_ref chain_end(vk_ref r) {
        int depth = 0;
        while (VK_REF_TYPE(r) == VK_T_XFORM) {
            if (VK_REF_INDEX(r) >= d->n_xforms) return bad(VK_ERR_INVALID, "xform index out of range"), VK_REF_NONE;
            if (++depth > VK_MAX_XFORM_DEPTH) return bad(VK_ERR_UNSUPPORTED, "wrapper chain deeper than VK_MAX_XFORM_DEPTH"), VK_REF_NONE;
            if (d->xforms[VK_REF_INDEX(r)].kind > VK_X_FLIP) return bad(VK_ERR_INVALID, "bad xform kind"), VK_REF_NONE;
            r = d->xforms[VK_REF_INDEX(r)].child;
        }
        return r;
    }
    bool medium_ok(vk_ref r, bool in_chain) {
        if (VK_REF_INDEX(r) >= d->n_media) return bad(VK_ERR_INVALID, "medium index out of range");
        const vk_medium& m = d->media[VK_REF_INDEX(r)];
        if (m.mat >= d->n_materials) return bad(VK_ERR_INVALID, "medium material out of range");
        vk_ref b = m.boundary;
        if (VK_REF_TYPE(b) == VK_T_XFORM) {
            if (in_chain) return bad(VK_ERR_UNSUPPORTED, "ConstantMedium with a transformed boundary inside another instance");
            b = chain_end(b);
            if (code != VK_OK) return false;
        }
        if (!is_leaf_type(VK_REF_TYPE(b)))
            return bad(VK_ERR_UNSUPPORTED, "ConstantMedium boundary must be a sphere, rect or box (optionally translated/rotated)");
        return leaf_ok(b);
    }
    // depth of the traversal stack needed below r; also fills node_medium
    int visit(vk_ref r, bool in_chain, bool& has_medium) {
        bool hx = false;
        return visit(r, in_chain, has_medium, hx);
    }
    int visit(vk_ref r, bool in_chain, bool& has_medium, bool& has_xform) {
        has_medium = false;
        has_xform = false;
        const uint32_t t = VK_REF_TYPE(r), i = VK_REF_INDEX(r);
        if (t == VK_T_NODE) {
            if (i >= d->n_nodes) return bad(VK_ERR_INVALID, "node index out of range"), 0;
            if (node_depth[i] == -1) return bad(VK_ERR_INVALID, "cycle in the BVH"), 0;
            if (node_depth[i] > 0) {
                // A sub-BVH shared between the world and an instance (a DAG) was validated for the frame it was first
                // reached in; below an instance it must not hold transforms (trav_prim_step keeps ONE instance frame).
                if (in_chain && node_xform[i])
                    return bad(VK_ERR_UNSUPPORTED, "nested instances (a shared sub-BVH holding a transform is also reached below a transform)"), 0;
                if (in_chain && !node_inchain[i]) node_inchain[i] = 1;
                has_medium = node_medium[i];
                has_xform = node_xform[i];
                return node_depth[i];
            }
            if (++level > 2 * VKD_STACK) return bad(VK_ERR_UNSUPPORTED, "BVH deeper than the traversal stack"), 0; // before the host stack suffers
            node_depth[i] = -1;
            bool ml = false, mr = false, xl = false, xr = false;
            const int dl = visit(d->nodes[i].left, in_chain, ml, xl);
            const int dr = d->nodes[i].right == d->nodes[i].left ? dl : visit(d->nodes[i].right, in_chain, mr, xr);
            --level;
            if (d->nodes[i].right == d->nodes[i].left) mr = ml;
            node_xform[i] = xl || xr;
            has_xform = node_xform[i];
            if (code != VK_OK) return 0;
            if (d->nodes[i].right == d->nodes[i].left && ml && VK_REF_TYPE(chain_end(d->nodes[i].left)) != VK_T_MEDIUM)
                return bad(VK_ERR_UNSUPPORTED, "single-object BVH leaf holding a medium inside a nested BVH"), 0;
            node_medium[i] = ml || mr;
            node_inchain[i] = in_chain;
            has_medium = node_medium[i];
            node_depth[i] = 1 + (dl > dr ? dl : dr);
            return node_depth[i];
        }
        if (t == VK_T_XFORM) {
            has_xform = true;
            if (in_chain) return bad(VK_ERR_UNSUPPORTED, "nested instances (a transform below another transform's BVH)"), 0;
            const vk_ref end = chain_end(r);
            if (code != VK_OK) return 0;
            if (VK_REF_TYPE(end) == VK_T_NODE) {
                bool hx = false;
                return 2 + visit(end, true, has_medium, hx);
            }
            if (VK_REF_TYPE(end) == VK_T_MEDIUM) {
                has_medium = true;
                medium_ok(end, true);
                return 1;
            }
            if (!is_leaf_type(VK_REF_TYPE(end))) return bad(VK_ERR_INVALID, "bad reference below a transform"), 0;
            leaf_ok(end);
            return 1;
        }
        if (t == VK_T_MEDIUM) {
            has_medium = true;
            medium_ok(r, in_chain);
            has_xform = i < d->n_media && VK_REF_TYPE(d->media[i].boundary) == VK_T_XFORM;
            return 1;
        }
        if (is_leaf_type(t)) {
            leaf_ok(r);
            return 1;
        }
        return bad(VK_ERR_INVALID, "bad hittable reference"), 0;
    }
    bool tex_has_image(uint32_t ti, int depth) {
        if (ti >= d->n_textures || depth > 16) return false;
        const vk_texture& t = d->textures[ti];
        if (t.type == VK_TEX_IMAGE) return true;
        if (t.type == VK_TEX_CHECKER) return tex_has_image(t.checker.odd, depth + 1) || tex_has_image(t.checker.even, depth + 1);
        return false;
    }
    bool run() {
        if (!d || d->api_version != VK_API_VERSION) return bad(VK_ERR_INVALID, "scene description: wrong api_version");
        for (uint32_t i = 0; i < d->n_textures; ++i) {
            const vk_texture& t = d->textures[i];
            if (t.type > VK_TEX_NOISE) return bad(VK_ERR_INVALID, "bad texture type");
            if (t.type == VK_TEX_CHECKER && (t.checker.odd >= d->n_textures || t.checker.even >= d->n_textures))
                return bad(VK_ERR_INVALID, "checker child out of range");
            if (t.type == VK_TEX_IMAGE && (t.image.width == 0 || t.image.height == 0 ||
                                           (uint64_t)t.image.texel_offset + (uint64_t)t.image.width * t.image.height * 3 > d->n_texel_bytes))
                return bad(VK_ERR_INVALID, "image texture outside the texel pool");
            if (t.type == VK_TEX_NOISE && t.noise.perlin >= d->n_perlins) return bad(VK_ERR_INVALID, "perlin index out of range");
        }
        for (uint32_t i = 0; i < d->n_materials; ++i) {
            const vk_material& m = d->materials[i];
            if (m.type > VK_M_SPECDIFFUSE) return bad(VK_ERR_INVALID, "bad material type");
            if (m.type == VK_M_SPECDIFFUSE) {
                if (m.tex >= d->n_materials || m.aux >= d->n_materials) return bad(VK_ERR_INVALID, "SpecDiffuse child out of range");
                if (d->materials[m.tex].type == VK_M_SPECDIFFUSE || d->materials[m.aux].type == VK_M_SPECDIFFUSE)
                    return bad(VK_ERR_UNSUPPORTED, "nested SpecDiffuse");
            } else if (m.type != VK_M_DIELECTRIC && m.tex >= d->n_textures)
                return bad(VK_ERR_INVALID, "material texture out of range");
        }
        for (uint32_t i = 0; i < d->n_spheres; ++i)
            if (d->sphere_mat[i] >= d->n_materials) return bad(VK_ERR_INVALID, "sphere material out of range");
        for (uint32_t i = 0; i < d->n_mspheres; ++i)
            if (d->mspheres[i].mat >= d->n_materials) return bad(VK_ERR_INVALID, "moving-sphere material out of range");
        for (uint32_t i = 0; i < d->n_rects; ++i) {
            const uint32_t ax = d->rects[i].axes;
            if (d->rects[i].mat >= d->n_materials) return bad(VK_ERR_INVALID, "rect material out of range");
            if ((ax & 3) > 2 || ((ax >> 2) & 3) > 2 || ((ax >> 4) & 3) > 2) return bad(VK_ERR_INVALID, "rect axis out of range");
        }
        for (uint32_t i = 0; i < d->n_boxes; ++i)
            if (d->boxes[i].mat >= d->n_materials) return bad(VK_ERR_INVALID, "box material out of range");
        if (d->n_nodes > VKD_INDEX(0xFFFFFFFFu) || d->n_spheres > VKD_INDEX(0xFFFFFFFFu)) return bad(VK_ERR_UNSUPPORTED, "too many primitives");
        // Every record, reachable from the root or not: the layout planner walks whole arrays (all xforms for the instanced
        // sub-BVHs, all nodes for the single-object leaves, all media), so a stray record with a wild reference must be
        // refused here, not only the ones the traversal below reaches (found by tests/sanitize_host.cpp under ASan).
        auto ref_ok = [&](vk_ref r) {
            const uint32_t t = VK_REF_TYPE(r), ix = VK_REF_INDEX(r);
            const uint32_t lim = t == VK_T_NODE ? d->n_nodes : t == VK_T_SPHERE ? d->n_spheres : t == VK_T_MSPHERE ? d->n_mspheres
                               : t == VK_T_RECT ? d->n_rects : t == VK_T_BOX ? d->n_boxes : t == VK_T_XFORM ? d->n_xforms
                               : t == VK_T_MEDIUM ? d->n_media : 0;
            return ix < lim;
        };
        for (uint32_t i = 0; i < d->n_nodes; ++i)
            if (!ref_ok(d->nodes[i].left) || !ref_ok(d->nodes[i].right)) return bad(VK_ERR_INVALID, "BVH node holds a reference out of range");
        for (uint32_t i = 0; i < d->n_xforms; ++i) {
            if (!ref_ok(d->xforms[i].child)) return bad(VK_ERR_INVALID, "transform holds a reference out of range");
            chain_end(VK_REF(VK_T_XFORM, i)); // kinds, and that the chain ends (a cycle of wrappers runs into the depth limit)
            if (code != VK_OK) return false;
        }
        for (uint32_t i = 0; i < d->n_media; ++i) {
            if (!ref_ok(d->media[i].boundary)) return bad(VK_ERR_INVALID, "medium boundary out of range");
            if (d->media[i].mat >= d->n_materials) return bad(VK_ERR_INVALID, "medium material out of range");
        }
        node_depth.assign(d->n_nodes, 0);
        node_medium.assign(d->n_nodes, 0);
        node_inchain.assign(d->n_nodes, 0);
        node_xform.assign(d->n_nodes, 0);
        level = 0;
        bool hm = false;
        const int depth = visit(d->root, false, hm);
        if (code != VK_OK) return false;
        if (depth + 2 > VKD_STACK) return bad(VK_ERR_UNSUPPORTED, "BVH deeper than the traversal stack");
        // an empty light list is accepted here: HEAD's integrator is refused at render time (the reference
        // panics, src/hittable.rs:431), the legacy integrator (VK_FLAG_LEGACY_SCATTER) does not use it
        for (uint32_t i = 0; i < d->n_lights; ++i) {
            const vk_ref l = d->lights[i];
            const uint32_t t = VK_REF_TYPE(l), ix = VK_REF_INDEX(l);
            const uint32_t lim = t == VK_T_NODE ? d->n_nodes : t == VK_T_SPHERE ? d->n_spheres : t == VK_T_MSPHERE ? d->n_mspheres
                               : t == VK_T_RECT ? d->n_rects : t == VK_T_BOX ? d->n_boxes : t == VK_T_XFORM ? d->n_xforms
                               : t == VK_T_MEDIUM ? d->n_media : 0;
            if (ix >= lim) return bad(VK_ERR_INVALID, "light reference out of range");
        }
        return true;
    }
};

// Unroll the reference's traversal into the typed batches of FlatProgram; false if the scene does not
// fit (then the BVH is traversed).
// A chain of wrapper ops (outermost first) composed into one affine map, object = R * world + t, in double.
// The reference applies the wrappers one after the other (src/hittable.rs:508, :591-595, :680-684, :769-773); composing
// them changes the rounding only, so only the render build uses the result.  out[0..8] = rows of R, out[9..11] = t.
inline void compose_flat_ops(const FlatOp* ops, size_t n, float* out) {
    double R[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}}, t[3] = {0, 0, 0};
    for (size_t k = 0; k < n; ++k) {
        const FlatOp& op = ops[k];
        if (op.kind == VKF_OP_TRANSLATE) { // subtracts its offset from the point in the frame reached so far
            t[0] -= op.a; t[1] -= op.b; t[2] -= op.c;
            continue;
        }
        // world -> object rotations of rot_fwd (vk_device.cuh): Y: x' = c x - s z, z' = s x + c z;
        // X: y' = c y + s z, z' = -s y + c z;  Z: x' = c x + s y, y' = -s x + c y
        const double sn = op.a, cs = op.b;
        double M[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
        if (op.kind == VKF_OP_ROTY) { M[0][0] = cs; M[0][2] = -sn; M[2][0] = sn; M[2][2] = cs; }
        else if (op.kind == VKF_OP_ROTX) { M[1][1] = cs; M[1][2] = sn; M[2][1] = -sn; M[2][2] = cs; }
        else { M[0][0] = cs; M[0][1] = sn; M[1][0] = -sn; M[1][1] = cs; }
        double R2[3][3], t2[3];
        for (int i = 0; i < 3; ++i) {
            t2[i] = M[i][0] * t[0] + M[i][1] * t[1] + M[i][2] * t[2];
            for (int j = 0; j < 3; ++j) R2[i][j] = M[i][0] * R[0][j] + M[i][1] * R[1][j] + M[i][2] * R[2][j];
        }
        for (int i = 0; i < 3; ++i) {
            t[i] = t2[i];
            for (int j = 0; j < 3; ++j) R[i][j] = R2[i][j];
        }
    }
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) out[3 * i + j] = (float)R[i][j];
        out[9 + i] = (float)t[i];
    }
}
// the ops of a wrapper chain, outermost first (FlipFace leaves the ray alone); returns the first non-wrapper child
inline vk_ref chain_ops(const vk_scene_desc* d, vk_ref r, std::vector<FlatOp>& ops) {
    while (VK_REF_TYPE(r) == VK_T_XFORM) {
        const vk_xform& x = d->xforms[VK_REF_INDEX(r)];
        if (x.kind == VK_X_TRANSLATE) ops.push_back(FlatOp{VKF_OP_TRANSLATE, x.a, x.b, x.c});
        else if (x.kind != VK_X_FLIP)
            ops.push_back(FlatOp{x.kind == VK_X_ROTATE_X ? (uint32_t)VKF_OP_ROTX : (x.kind == VK_X_ROTATE_Y ? (uint32_t)VKF_OP_ROTY : (uint32_t)VKF_OP_ROTZ), x.a, x.b, 0.f});
        r = x.child;
    }
    return r;
}

struct FlatBuilder {
    const vk_scene_desc* d;
    struct Seg {
        std::vector<FlatOp> ops;
        std::vector<std::pair<FlatRect, FlatHit>> rects[6];
        std::vector<std::pair<FlatSphere, FlatHit>> sph, msph;
        std::vector<FlatHit> med;
        std::vector<uint32_t> bvh; // roots of homogeneous subtrees kept as BVHs (hybrid program)
        struct Box {
            float mn[3], mx[3];
            size_t at[3]; // position of sides 0, 2, 4 in rects[3], rects[4], rects[5] (sides 1, 3, 5 follow them)
        };
        std::vector<Box> boxes;
        uint32_t inst = 0;
    };
    std::vector<Seg> segs;
    // hybrid mode: a subtree whose leaves are all of ONE plain primitive kind (no wrapper, no medium) and
    // that holds more than VKF_SUBTREE_MIN of them stays a BVH; only the mixed top of the tree is unrolled
    bool hybrid = false;
    struct NodeInfo {
        uint32_t leaves = 0;
        uint8_t kind = 0; // VK_T_* shared by every leaf below, 0xFF = mixed / wrapper / medium
        bool done = false;
    };
    std::vector<NodeInfo> info;
    NodeInfo classify(vk_ref r) {
        NodeInfo out;
        const uint32_t t = VK_REF_TYPE(r);
        if (t != VK_T_NODE) {
            out.leaves = 1;
            out.kind = (t == VK_T_SPHERE || t == VK_T_RECT || t == VK_T_BOX) ? (uint8_t)t : (uint8_t)0xFF;
            return out;
        }
        NodeInfo& me = info[VK_REF_INDEX(r)];
        if (me.done) return me;
        const vk_node& n = d->nodes[VK_REF_INDEX(r)];
        const NodeInfo a = classify(n.left), b = n.right == n.left ? a : classify(n.right);
        me.leaves = a.leaves + (n.right == n.left ? 0 : b.leaves);
        me.kind = (a.kind == b.kind) ? a.kind : (uint8_t)0xFF;
        me.done = true;
        return me;
    }

    bool rect(Seg& g, float c0, float c1, float d0, float d1, float k, uint32_t axes, vk_ref ref, uint32_t face, bool box_side) {
        const uint32_t a0 = axes & 3u, a1 = (axes >> 2) & 3u, a2 = (axes >> 4) & 3u;
        // the canonical axis order of Rect::XYRect/XZRect/YZRect (src/hittable.rs:214-226) is assumed
        const bool canonical = (a2 == 2 && a0 == 0 && a1 == 1) || (a2 == 1 && a0 == 0 && a1 == 2) || (a2 == 0 && a0 == 1 && a1 == 2);
        if (!canonical) return false;
        FlatRect e{};
        e.bounds = make_float4(c0, c1, d0, d1);
        e.k = k;

        FlatHit h{ref, g.inst, face, 0u};
        g.rects[(a2 == 2 ? 0 : (a2 == 1 ? 1 : 2)) + (box_side ? 3 : 0)].push_back({e, h});
        return true;
    }
    size_t n_emitted = 0; // entries so far: a scene that cannot fit is abandoned early, not walked to the end
    bool emit(vk_ref ref, size_t si, uint32_t dup) {
        if (++n_emitted > 4 * (VKF_MAX_RECTS + VKF_MAX_SPHERES + VKF_MAX_MEDIA + VKF_MAX_BVH + VKF_MAX_OPS)) return false;
        const uint32_t i = VK_REF_INDEX(ref);
        switch (VK_REF_TYPE(ref)) {
        case VK_T_NODE: {
            if (hybrid) {
                const NodeInfo ni = classify(ref);
                if (ni.kind != 0xFF && ni.leaves > 8) { // homogeneous and worth a BVH: keep it as one entry
                    segs[si].bvh.push_back(ref);
                    return true;
                }
            }
            const vk_node& n = d->nodes[i];
            if (!emit(n.left, si, dup)) return false;
            if (n.right != n.left) return emit(n.right, si, dup);
            vk_ref end = n.left; // single-object leaf: the second visit only matters for a medium
            while (VK_REF_TYPE(end) == VK_T_XFORM) end = d->xforms[VK_REF_INDEX(end)].child;
            return VK_REF_TYPE(end) == VK_T_MEDIUM ? emit(n.left, si, VKD_DUP) : true;
        }
        case VK_T_SPHERE: {
            FlatSphere e{};
            e.a = make_float4(d->spheres[i].center[0], d->spheres[i].center[1], d->spheres[i].center[2], d->spheres[i].radius);
            segs[si].sph.push_back({e, FlatHit{ref, segs[si].inst, 0u, 0u}});
            return true;
        }
        case VK_T_MSPHERE: {
            const vk_msphere& m = d->mspheres[i];
            FlatSphere e{};
            e.a = make_float4(m.center0[0], m.center0[1], m.center0[2], m.radius);
            e.b = make_float4(m.center1[0], m.center1[1], m.center1[2], m.time0);
            e.time1 = m.time1;
            segs[si].msph.push_back({e, FlatHit{ref, segs[si].inst, 0u, 0u}});
            return true;
        }
        case VK_T_RECT: {
            const vk_rect& r = d->rects[i];
            return rect(segs[si], r.c0, r.c1, r.d0, r.d1, r.k, r.axes, ref, 0, false);
        }
        case VK_T_BOX: { // the six sides in Boxy::new order (src/hittable.rs:325-353)
            const vk_box& b = d->boxes[i];
            const float* mn = b.box_min;
            const float* mx = b.box_max;
            const uint32_t XY = 0u | (1u << 2) | (2u << 4), XZ = 0u | (2u << 2) | (1u << 4), YZ = 1u | (2u << 2) | (0u << 4);
            Seg& g = segs[si];
            g.boxes.push_back({{mn[0], mn[1], mn[2]}, {mx[0], mx[1], mx[2]}, {g.rects[3].size(), g.rects[4].size(), g.rects[5].size()}});
            return rect(g, mn[0], mx[0], mn[1], mx[1], mx[2], XY, ref, 0, true) && rect(g, mn[0], mx[0], mn[1], mx[1], mn[2], XY, ref, 1, true) &&
                   rect(g, mn[0], mx[0], mn[2], mx[2], mx[1], XZ, ref, 2, true) && rect(g, mn[0], mx[0], mn[2], mx[2], mn[1], XZ, ref, 3, true) &&
                   rect(g, mn[1], mx[1], mn[2], mx[2], mx[0], YZ, ref, 4, true) && rect(g, mn[1], mx[1], mn[2], mx[2], mn[0], YZ, ref, 5, true);
        }
        case VK_T_MEDIUM:
            segs[si].med.push_back(FlatHit{ref | dup, segs[si].inst, 0u, 0u});
            return true;
        case VK_T_XFORM: {
            if (si != 0) return false; // nested instances are refused by the validator anyway
            Seg g;
            g.inst = ref; // instance id = outermost wrapper
            const vk_ref r = chain_ops(d, ref, g.ops); // (FlipFace leaves the ray alone; the flip happens in resolve_hit)
            segs.push_back(std::move(g));
            return emit(r, segs.size() - 1, dup);
        }
        default: return false;
        }
    }
    bool build(FlatProgram* P, bool hybrid_mode) {
        *P = FlatProgram{};
        hybrid = hybrid_mode;
        n_emitted = 0;
        info.assign(hybrid ? d->n_nodes : 0, NodeInfo{});
        segs.clear();
        segs.emplace_back();
        if (!emit(d->root, 0, 0)) return false;
        if (segs.size() > VKF_MAX_SEGS) return false;
        uint32_t n_ops = 0, n_rects = 0, n_sph = 0, n_hits = 0, n_med = 0, n_bvh = 0, n_boxes = 0;
        for (size_t s = 0; s < segs.size(); ++s) {
            Seg& g = segs[s];
            FlatSeg& o = P->segs[s];
            if (n_ops + g.ops.size() > VKF_MAX_OPS) return false;
            o.op0 = (uint8_t)n_ops;
            for (const FlatOp& op : g.ops) P->ops[n_ops++] = op;
            o.op1 = (uint8_t)n_ops;
            for (int k = 0; k < 6; ++k) {
                if (n_rects + g.rects[k].size() > VKF_MAX_RECTS) return false;
                o.rect0[k] = (uint8_t)n_rects;
                for (auto& e : g.rects[k]) {
                    e.first.hit = n_hits;
                    P->hits[n_hits++] = e.second;
                    P->rects[n_rects++] = e.first;
                }
                o.rect1[k] = (uint8_t)n_rects;
            }
            if (n_boxes + g.boxes.size() > VKF_MAX_BOXES) return false;
            o.box0 = (uint8_t)n_boxes;
            for (const Seg::Box& b : g.boxes) { // (the sides' hit entries were numbered just above)
                const uint32_t hz = g.rects[3][b.at[0]].first.hit, hy = g.rects[4][b.at[1]].first.hit, hx = g.rects[5][b.at[2]].first.hit;
                FlatBox& fb = P->boxes[n_boxes++];
                fb.mn = make_float4(b.mn[0], b.mn[1], b.mn[2], __uint_as_float_host(hz));
                fb.mx = make_float4(b.mx[0], b.mx[1], b.mx[2], __uint_as_float_host(hy | (hx << 16)));
            }
            o.box1 = (uint8_t)n_boxes;
            if (n_sph + g.sph.size() + g.msph.size() > VKF_MAX_SPHERES) return false;
            o.sph0 = (uint8_t)n_sph;
            for (auto& e : g.sph) {
                e.first.hit = n_hits;
                P->hits[n_hits++] = e.second;
                P->spheres[n_sph++] = e.first;
            }
            o.sph1 = o.msph0 = (uint8_t)n_sph;
            for (auto& e : g.msph) {
                e.first.hit = n_hits;
                P->hits[n_hits++] = e.second;
                P->spheres[n_sph++] = e.first;
            }
            o.msph1 = (uint8_t)n_sph;
            if (n_med + g.med.size() > VKF_MAX_MEDIA) return false;
            o.med0 = (uint8_t)n_hits;
            P->seg_fm0[s] = (uint8_t)n_med;
            for (const FlatHit& h : g.med) {
                FlatMedium& fm = P->fmed[n_med];
                fm = FlatMedium{};
                const vk_medium& md = d->media[VK_REF_INDEX(h.prim & ~VKD_DUP)];
                std::vector<FlatOp> ops;
                const vk_ref leaf = chain_ops(d, md.boundary, ops);
                compose_flat_ops(ops.data(), ops.size(), fm.aff);
                if (VK_REF_TYPE(leaf) == VK_T_BOX) {
                    const vk_box& b = d->boxes[VK_REF_INDEX(leaf)];
                    fm.mn = make_float4(b.box_min[0], b.box_min[1], b.box_min[2], md.neg_inv_density);
                    fm.mx = make_float4(b.box_max[0], b.box_max[1], b.box_max[2], __uint_as_float_host(1u | (ops.empty() ? 0u : 2u)));
                }
                P->hits[n_hits++] = h;
                ++n_med;
            }
            o.med1 = (uint8_t)n_hits;
            if (n_bvh + g.bvh.size() > VKF_MAX_BVH) return false;
            o.bvh0 = (uint8_t)n_bvh;
            for (uint32_t r : g.bvh) P->bvh[n_bvh++] = r;
            o.bvh1 = (uint8_t)n_bvh;
            P->seg_inst[s] = g.inst;
            compose_flat_ops(g.ops.data(), g.ops.size(), P->seg_affine[s]);
        }
        P->n_bvh = n_bvh;
        for (uint32_t h = 0; h < n_hits; ++h) { // shading class of each entry's material
            const vk_ref pr = P->hits[h].prim & ~VKD_DUP;
            const uint32_t i = VK_REF_INDEX(pr);
            uint32_t mat = 0;
            switch (VK_REF_TYPE(pr)) {
            case VK_T_SPHERE: mat = d->sphere_mat[i]; break;
            case VK_T_MSPHERE: mat = d->mspheres[i].mat; break;
            case VK_T_RECT: mat = d->rects[i].mat; break;
            case VK_T_BOX: mat = d->boxes[i].mat; break;
            case VK_T_MEDIUM: mat = d->media[i].mat; break;
            default: return false;
            }
            const uint32_t t = d->materials[mat].type;
            P->hits[h].cls = t == VK_M_DIFFUSE_LIGHT ? 0u : t == VK_M_DIELECTRIC ? 1u : t == VK_M_METAL ? 2u : 3u;
        }
        static_assert(VKF_MAX_RECTS + VKF_MAX_SPHERES + VKF_MAX_MEDIA <= 256, "class-tagged ids keep the entry in 8 bits");
        auto tagged = [&](uint32_t h) { return VKF_HITC(h, P->hits[h].cls, P->hits[h].inst); };
        for (uint32_t i = 0; i < n_rects; ++i) P->rects[i].hitc = tagged(P->rects[i].hit);
        for (uint32_t i = 0; i < n_sph; ++i) P->spheres[i].hitc = tagged(P->spheres[i].hit);
        for (uint32_t i = 0; i < n_boxes; ++i) { // (a Boxy has one material: its six sides share the class)
            const uint32_t hz = __float_as_uint_host(P->boxes[i].mn.w), hyx = __float_as_uint_host(P->boxes[i].mx.w);
            P->boxes[i].mn.w = __uint_as_float_host(tagged(hz));
            P->boxes[i].mx.w = __uint_as_float_host(tagged(hyx & 0xFFFFu) | (tagged(hyx >> 16) << 16));
        }
        P->n_segs = (uint32_t)segs.size();
        P->n = n_hits + n_bvh;
        return P->n > 0;
    }
};

// Host-side re-layout of a validated scene (no device needed): the node array with single-object
// leaves resolved, the 4-wide nodes, the flat program and the "simple scene" test.  vk_scene_upload
// copies the results to the device; vk_scene_check reports them so that CPU tests can cover this code.
struct Relayout {
    std::vector<vk_node> nodes;
    std::vector<float4> wnodes;
    FlatProgram flat{};
    uint32_t levels_world = 0, levels_sub = 0, n_wide = 0, stack_need = 0;
    bool simple = false, has_specdiffuse = false;
    uint32_t flat_shape = VKF_SHAPE_NONE; // the compiled shape the program has (flat_static_shape), if any
    // Per entry of the flat program's hit table, for the render build's shade stage: {world-space outward normal,
    // flags} {material index, -, -, -}.  flags bit 0: the HitRec of this entry can be written down directly --
    // p = o + t d, normal = the constant normal turned against the ray -- instead of walking its wrapper chain; bit 1:
    // FlipFace.  That holds for a rect or box side whose material reads no (u, v), and which either sits in the world
    // frame, or under a chain whose OUTERMOST wrapper is a Translate and whose material does not read `front`
    // (Lambertian, Metal, Isotropic): every level of the chain re-runs set_face_normal (src/hittable.rs:519, :618), so
    // what leaves the Translate is +-(the rotated axis), turned against the WORLD ray -- whatever the levels below
    // did (SURVEY Q9).  `front` of a plain rect is dot(d, n) < 0, flipped by FlipFace (:300-308).
    std::vector<float4> flat_shade;
    // Per ConstantMedium, for the render build's medium_t: 4 x float4 = the three rows {R | t} of the boundary's wrapper
    // chain composed into one affine map, then {boundary leaf, chain present, -, -}.
    std::vector<float4> media_plan;
    // returns nullptr or the reason the scene is unsupported
    const char* run(const vk_scene_desc* d) {
    // GPU-side re-layout of the node array: a single-object leaf (left == right) is tested twice
        // by the reference; that only matters for a ConstantMedium (two free-flight draws), so the
        // second visit is kept (flagged) only there and dropped for deterministic primitives.
        nodes.assign(d->nodes, d->nodes + d->n_nodes);
        for (uint32_t i = 0; i < d->n_nodes; ++i)
            if (nodes[i].left == nodes[i].right) {
                vk_ref end = nodes[i].left;
                while (VK_REF_TYPE(end) == VK_T_XFORM) end = d->xforms[VK_REF_INDEX(end)].child;
                nodes[i].right = VK_REF_TYPE(end) == VK_T_MEDIUM ? (nodes[i].left | VKD_DUP) : VK_REF_NONE;
            }
        // 4-wide nodes from the reference's binary tree (see DScene): start from a node's two children and
        // keep opening the inner child with the largest surface area until four slots are filled.
        wnodes.assign((size_t)d->n_nodes * 8, make_float4(0, 0, 0, 0));
        {
            struct Slot {
                vk_ref ref;
                float mn[3], mx[3];
            };
            std::vector<uint8_t> built(d->n_nodes, 0);
            std::vector<uint32_t> todo, level(d->n_nodes, 0); // level: 4-wide levels above the node inside its BVH
            levels_world = levels_sub = 0;
            bool in_sub = false;
            auto want = [&](vk_ref r, uint32_t lvl) {
                if (VK_REF_TYPE(r) == VK_T_NODE && !built[VK_REF_INDEX(r)]) {
                    built[VK_REF_INDEX(r)] = 1;
                    level[VK_REF_INDEX(r)] = lvl;
                    todo.push_back(VK_REF_INDEX(r));
                    uint32_t& top = in_sub ? levels_sub : levels_world;
                    if (lvl + 1 > top) top = lvl + 1;
                }
            };
            auto child_slot = [&](vk_ref r, const vk_node& parent) { // a node child brings its own box, a primitive its parent's
                const vk_node& b = VK_REF_TYPE(r) == VK_T_NODE ? d->nodes[VK_REF_INDEX(r)] : parent;
                Slot s{r, {b.bb_min[0], b.bb_min[1], b.bb_min[2]}, {b.bb_max[0], b.bb_max[1], b.bb_max[2]}};
                return s;
            };
            auto area = [](const Slot& s) {
                const float x = s.mx[0] - s.mn[0], y = s.mx[1] - s.mn[1], z = s.mx[2] - s.mn[2];
                return x * y + y * z + z * x;
            };
            // the world's BVH first, then the instanced sub-BVHs (an instance is never nested: see Validator)
            for (int pass = 0; pass < 2; ++pass) {
            in_sub = pass == 1;
            if (pass == 0) want(d->root, 0);
            else
                for (uint32_t i = 0; i < d->n_xforms; ++i) want(d->xforms[i].child, 0);
            while (!todo.empty()) {
                const uint32_t ni = todo.back();
                todo.pop_back();
                Slot slots[6]; // never more than four after a round; two are added before one is removed
                size_t n_slots = 0;
                auto add_children = [&](uint32_t n) {
                    if (nodes[n].left != VK_REF_NONE) slots[n_slots++] = child_slot(nodes[n].left, d->nodes[n]);
                    if (nodes[n].right != VK_REF_NONE) slots[n_slots++] = child_slot(nodes[n].right, d->nodes[n]);
                };
                add_children(ni);
                while (n_slots < 4) {
                    int best = -1;
                    for (size_t k = 0; k < n_slots; ++k)
                        if (VK_REF_TYPE(slots[k].ref) == VK_T_NODE) {
                            const uint32_t n = VK_REF_INDEX(slots[k].ref);
                            const size_t kids = (nodes[n].left != VK_REF_NONE) + (nodes[n].right != VK_REF_NONE);
                            if (n_slots - 1 + kids > 4) continue;
                            if (best < 0 || area(slots[k]) > area(slots[best])) best = (int)k;
                        }
                    if (best < 0) break;
                    const uint32_t n = VK_REF_INDEX(slots[best].ref);
                    for (size_t k = (size_t)best; k + 1 < n_slots; ++k) slots[k] = slots[k + 1];
                    --n_slots;
                    add_children(n);
                }
                ++n_wide;
                float4* q = &wnodes[(size_t)ni * 8];
                float* f = reinterpret_cast<float*>(q);
                for (size_t k = 0; k < 4; ++k) {
                    const bool have = k < n_slots;
                    for (int ax = 0; ax < 3; ++ax) {
                        f[(2 * ax) * 4 + k] = have ? slots[k].mn[ax] : 0.f;
                        f[(2 * ax + 1) * 4 + k] = have ? slots[k].mx[ax] : 0.f;
                    }
                    f[6 * 4 + k] = __uint_as_float_host(have ? slots[k].ref : VK_REF_NONE);
                    if (have) want(slots[k].ref, level[ni] + 1);
                }
            }
            }
            // a visit pushes at most three siblings; an instance adds its exit marker
            if (3 * levels_world + 1 + 3 * levels_sub + 2 > VKD_STACK)
                return "BVH deeper than the traversal stack";
        }
        stack_need = 3 * levels_world + 1 + 3 * levels_sub + 2;
        // the whole scene as typed batches if it is small; else, for a heterogeneous scene (wrappers or media
        // present), the mixed top of the tree as batches and its homogeneous subtrees as BVH entries
        FlatBuilder fb;
        fb.d = d;
        if (!fb.build(&flat, false)) {
            const bool heterogeneous = d->n_media > 0 || d->n_xforms > 0;
            // Off by default: measured on the final scene (800x800x64) the hybrid program renders in 52.5 ms
            // against 50.0 ms for the plain 4-wide BVH -- the flat top tests all nine loose objects (two
            // media included) for every ray where the BVH culls some, and the subtree traversals keep their
            // divergence.  VECCHIO_HYBRID=1 enables it (parity-tested: same image bit for bit).
            const char* hy = std::getenv("VECCHIO_HYBRID");
            if (!(heterogeneous && !(hy && hy[0] == '0') && fb.build(&flat, true) && flat.n_bvh > 0)) flat = FlatProgram{};
        }
        media_plan.assign(4 * (size_t)d->n_media, make_float4(0, 0, 0, 0));
        for (uint32_t i = 0; i < d->n_media; ++i) {
            std::vector<FlatOp> ops;
            const vk_ref leaf = chain_ops(d, d->media[i].boundary, ops);
            float m[12];
            compose_flat_ops(ops.data(), ops.size(), m);
            for (int r = 0; r < 3; ++r) media_plan[4 * i + r] = make_float4(m[3 * r], m[3 * r + 1], m[3 * r + 2], m[9 + r]);
            media_plan[4 * i + 3] = make_float4(__uint_as_float_host(leaf), __uint_as_float_host(ops.empty() ? 0u : 1u), 0.f, 0.f);
        }
        flat_shade.clear();
        if (flat.n && flat.n_bvh == 0) {
            Validator tv;
            tv.d = d;
            flat_shade.assign(2 * (size_t)flat.n, make_float4(0, 0, 0, 0));
            for (uint32_t h = 0; h < flat.n; ++h) {
                const FlatHit& fh = flat.hits[h];
                const vk_ref pr = fh.prim & ~VKD_DUP;
                const uint32_t i = VK_REF_INDEX(pr);
                uint32_t a2, flip, mat;
                // every entry: {-, leaf, instance | face << 28 | has-instance << 31, -}: what the shade stage hands to resolve_hit
                // when the HitRec cannot be written down directly (the slot only keeps the distance and the entry)
                flat_shade[2 * h + 1] = make_float4(0.f, __uint_as_float_host(pr),
                                                    __uint_as_float_host((fh.inst ? (0x80000000u | VKD_INDEX(fh.inst)) : 0u) | (fh.face << 28)), 0.f);
                if (VK_REF_TYPE(pr) == VK_T_RECT) {
                    a2 = (d->rects[i].axes >> 4) & 3u;
                    flip = (d->rects[i].axes & VK_RECT_FLIP) ? 1u : 0u;
                    mat = d->rects[i].mat;
                } else if (VK_REF_TYPE(pr) == VK_T_BOX) { // side `face` of Boxy::new: z, z, y, y, x, x; odd ones wrapped in FlipFace
                    a2 = fh.face < 2 ? 2u : (fh.face < 4 ? 1u : 0u);
                    flip = fh.face & 1u;
                    mat = d->boxes[i].mat;
                } else
                    continue;
                const vk_material& m = d->materials[mat];
                const bool reads_uv = m.type == VK_M_SPECDIFFUSE || (m.type != VK_M_DIELECTRIC && tv.tex_has_image(m.tex, 0));
                const bool reads_front = m.type == VK_M_DIELECTRIC || m.type == VK_M_DIFFUSE_LIGHT || m.type == VK_M_SPECDIFFUSE;
                float n[3] = {a2 == 0 ? 1.f : 0.f, a2 == 1 ? 1.f : 0.f, a2 == 2 ? 1.f : 0.f};
                bool ok = !reads_uv;
                if (fh.inst) { // walk the chain, collect the levels, rotate the normal back out (innermost level first)
                    std::vector<vk_xform> chain;
                    vk_ref r = fh.inst;
                    while (VK_REF_TYPE(r) == VK_T_XFORM) {
                        chain.push_back(d->xforms[VK_REF_INDEX(r)]);
                        r = chain.back().child;
                    }
                    ok = ok && !reads_front && !chain.empty() && chain.front().kind == VK_X_TRANSLATE;
                    for (size_t l = chain.size(); l-- > 0 && ok;) {
                        const vk_xform& x = chain[l];
                        const float sn = x.a, cs = x.b, v0 = n[0], v1 = n[1], v2 = n[2];
                        if (x.kind == VK_X_ROTATE_Y) { n[0] = cs * v0 + sn * v2; n[2] = -sn * v0 + cs * v2; }          // rot_back, vk_device.cuh
                        else if (x.kind == VK_X_ROTATE_X) { n[1] = cs * v1 - sn * v2; n[2] = sn * v1 + cs * v2; }
                        else if (x.kind == VK_X_ROTATE_Z) { n[0] = cs * v0 - sn * v1; n[1] = sn * v0 + cs * v1; }
                        else if (x.kind == VK_X_FLIP) ok = false; // FlipFace of a non-rect inside a chain: keep the general path
                    }
                }
                if (!ok) continue;
                flat_shade[2 * h] = make_float4(n[0], n[1], n[2], __uint_as_float_host(1u | (flip << 1)));
                flat_shade[2 * h + 1].x = __uint_as_float_host(mat);
            }
        }
        flat_shape = flat_static_shape(flat);
        has_specdiffuse = false;
        for (uint32_t i = 0; i < d->n_materials; ++i) has_specdiffuse |= d->materials[i].type == VK_M_SPECDIFFUSE;
        // simple: solid textures only; Lambertian / Dielectric / DiffuseLight / Isotropic only; no moving sphere;
        // exactly one light, an unflipped Rect
        simple = d->n_mspheres == 0 && d->n_lights == 1 && VK_REF_TYPE(d->lights[0]) == VK_T_RECT &&
                 !(d->rects[VK_REF_INDEX(d->lights[0])].axes & VK_RECT_FLIP);
        for (uint32_t i = 0; i < d->n_textures && simple; ++i) simple = d->textures[i].type == VK_TEX_SOLID;
        for (uint32_t i = 0; i < d->n_materials && simple; ++i)
            simple = d->materials[i].type == VK_M_LAMBERTIAN || d->materials[i].type == VK_M_DIELECTRIC ||
                     d->materials[i].type == VK_M_DIFFUSE_LIGHT || d->materials[i].type == VK_M_ISOTROPIC;
        return nullptr;
    }
};


} // namespace vkhost
