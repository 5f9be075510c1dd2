// vk_relayout.cu -- vk_scene_check: the validator and the layout planner of vk_relayout.h behind the C ABI,
// without a device (what the CPU tests exercise).
#include <cstdio>
#include <cstdlib>

#include "vk_relayout.h"

using namespace vkhost;

extern "C" {

int vk_scene_check(const vk_scene_desc* d, vk_scene_info* info, char* err, size_t err_len) {
    auto report = [&](int code, const std::string& msg) {
        if (err && err_len) std::snprintf(err, err_len, "%s", msg.c_str());
        return code;
    };
    if (!d) return report(VK_ERR_INVALID, "null scene");
    Validator v;
    v.d = d;
    if (!v.run()) return report(v.code, v.err);
    Relayout R;
    if (const char* why = R.run(d)) return report(VK_ERR_UNSUPPORTED, why);
    if (info) {
        info->flat_entries = R.flat.n;
        info->flat_segments = R.flat.n ? R.flat.n_segs : 0;
        info->flat_subtrees = R.flat.n ? R.flat.n_bvh : 0;
        info->simple = R.simple ? 1u : 0u;
        info->wide_nodes = R.n_wide;
        info->stack_need = R.stack_need;
        info->wide_levels_world = R.levels_world;
        info->wide_levels_instance = R.levels_sub;
        info->dynamic_megakernel = d->n_nodes >= 65536u ? 1u : 0u;
        info->flat_boxes = 0;
        for (uint32_t s = 0; R.flat.n && s < R.flat.n_segs; ++s) info->flat_boxes += R.flat.segs[s].box1 - R.flat.segs[s].box0;
        info->flat_shape = R.flat_shape;
        info->flat_direct = 0;
        for (size_t h = 0; 2 * h + 1 < R.flat_shade.size(); ++h) info->flat_direct += __float_as_uint_host(R.flat_shade[2 * h].w) & 1u;
    }
    if (err && err_len) err[0] = 0;
    return VK_OK;
}

} // extern "C"
