"""ctypes mirror of include/vecchio_gpu.h and include/vecchio_host.h (structs only)."""
import ctypes as C

VK_API_VERSION = 1
VK_OK = 0
VK_ERR_INVALID, VK_ERR_NO_DEVICE, VK_ERR_CUDA, VK_ERR_UNSUPPORTED, VK_ERR_NO_SCENE, VK_ERR_OOM = -1, -2, -3, -4, -5, -6

VK_T_NONE, VK_T_NODE, VK_T_SPHERE, VK_T_MSPHERE, VK_T_RECT, VK_T_BOX, VK_T_XFORM, VK_T_MEDIUM = range(8)
VK_VARIANT_AUTO, VK_VARIANT_MEGAKERNEL, VK_VARIANT_WAVEFRONT, VK_VARIANT_STAGED, VK_VARIANT_WARPQ, VK_VARIANT_STEPQ = 0, 1, 2, 3, 4, 5
VK_FLAG_STRICT_MATH = 1
VK_FLAG_FORCE_BVH = 2
VK_FLAG_LEGACY_SCATTER = 4
VK_FLAG_SKY_BACKGROUND = 8
VK_MEDIUM_XI_SLOTS = 8
VK_EVAL_BOUNCE, VK_EVAL_BOUNCE_LEGACY, VK_EVAL_TEXTURE, VK_EVAL_LIGHTS_PDF, VK_EVAL_LIGHT_RANDOM = range(5)
VK_M_LAMBERTIAN, VK_M_METAL, VK_M_DIELECTRIC, VK_M_DIFFUSE_LIGHT, VK_M_ISOTROPIC, VK_M_SPECDIFFUSE = range(6)
VK_TEX_SOLID, VK_TEX_CHECKER, VK_TEX_IMAGE, VK_TEX_NOISE = range(4)
VK_RECT_FLIP = 0x100


def ref_type(r):
    return (int(r) >> 28) & 0xF


def ref_index(r):
    return int(r) & 0x0FFFFFFF


class vk_node(C.Structure):
    _fields_ = [("bb_min", C.c_float * 3), ("left", C.c_uint32), ("bb_max", C.c_float * 3), ("right", C.c_uint32)]


class vk_sphere(C.Structure):
    _fields_ = [("center", C.c_float * 3), ("radius", C.c_float)]


class vk_msphere(C.Structure):
    _fields_ = [("center0", C.c_float * 3), ("radius", C.c_float), ("center1", C.c_float * 3), ("time0", C.c_float),
                ("time1", C.c_float), ("mat", C.c_uint32), ("_pad", C.c_uint32 * 2)]


class vk_rect(C.Structure):
    _fields_ = [("c0", C.c_float), ("c1", C.c_float), ("d0", C.c_float), ("d1", C.c_float), ("k", C.c_float),
                ("axes", C.c_uint32), ("mat", C.c_uint32), ("_pad", C.c_uint32)]


class vk_box(C.Structure):
    _fields_ = [("box_min", C.c_float * 3), ("mat", C.c_uint32), ("box_max", C.c_float * 3), ("_pad", C.c_uint32)]


class vk_xform(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("child", C.c_uint32), ("_pad0", C.c_uint32 * 2), ("a", C.c_float),
                ("b", C.c_float), ("c", C.c_float), ("_pad1", C.c_uint32)]


class vk_medium(C.Structure):
    _fields_ = [("boundary", C.c_uint32), ("neg_inv_density", C.c_float), ("mat", C.c_uint32), ("_pad", C.c_uint32)]


class vk_material(C.Structure):
    _fields_ = [("type", C.c_uint32), ("tex", C.c_uint32), ("param", C.c_float), ("aux", C.c_uint32)]


class vk_texture(C.Structure):
    _fields_ = [("type", C.c_uint32), ("w", C.c_uint32 * 3)]  # union payload viewed as 3 words


class vk_perlin(C.Structure):
    _fields_ = [("ranvec", (C.c_float * 3) * 256), ("perm_x", C.c_uint8 * 256), ("perm_y", C.c_uint8 * 256),
                ("perm_z", C.c_uint8 * 256)]


class vk_scene_desc(C.Structure):
    _fields_ = [
        ("api_version", C.c_uint32), ("root", C.c_uint32),
        ("nodes", C.POINTER(vk_node)), ("n_nodes", C.c_uint32),
        ("spheres", C.POINTER(vk_sphere)), ("sphere_mat", C.POINTER(C.c_uint32)), ("n_spheres", C.c_uint32),
        ("mspheres", C.POINTER(vk_msphere)), ("n_mspheres", C.c_uint32),
        ("rects", C.POINTER(vk_rect)), ("n_rects", C.c_uint32),
        ("boxes", C.POINTER(vk_box)), ("n_boxes", C.c_uint32),
        ("xforms", C.POINTER(vk_xform)), ("n_xforms", C.c_uint32),
        ("media", C.POINTER(vk_medium)), ("n_media", C.c_uint32),
        ("lights", C.POINTER(C.c_uint32)), ("n_lights", C.c_uint32),
        ("materials", C.POINTER(vk_material)), ("n_materials", C.c_uint32),
        ("textures", C.POINTER(vk_texture)), ("n_textures", C.c_uint32),
        ("texels", C.POINTER(C.c_uint8)), ("n_texel_bytes", C.c_uint64),
        ("perlins", C.POINTER(vk_perlin)), ("n_perlins", C.c_uint32),
    ]


class vk_camera(C.Structure):
    _fields_ = [("origin", C.c_float * 3), ("lower_left_corner", C.c_float * 3), ("horizontal", C.c_float * 3),
                ("vertical", C.c_float * 3), ("u", C.c_float * 3), ("v", C.c_float * 3), ("w", C.c_float * 3),
                ("lens_radius", C.c_float), ("time0", C.c_float), ("time1", C.c_float)]


class vk_render_params(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("spp", C.c_uint32), ("spp_begin", C.c_uint32),
                ("spp_count", C.c_uint32), ("max_depth", C.c_uint32), ("seed", C.c_uint64),
                ("background", C.c_float * 3), ("variant", C.c_uint32), ("flags", C.c_uint32)]


class vk_stats(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("rays", C.c_uint64), ("dropped_samples", C.c_uint64),
                ("ms_kernels", C.c_float), ("ms_total", C.c_float), ("variant", C.c_uint32), ("launches", C.c_uint32),
                ("node_visits", C.c_uint64), ("prim_tests", C.c_uint64)]


class vk_scene_info(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("flat_entries", "flat_segments", "flat_subtrees", "simple", "wide_nodes", "wide_levels_world",
                                          "wide_levels_instance", "stack_need", "dynamic_megakernel", "flat_boxes", "flat_direct", "flat_shape")]


class vk_ray(C.Structure):
    _fields_ = [("origin", C.c_float * 3), ("direction", C.c_float * 3), ("time", C.c_float), ("tmin", C.c_float),
                ("tmax", C.c_float)]


class vk_hit(C.Structure):
    _fields_ = [("prim", C.c_uint32), ("face", C.c_uint32), ("mat", C.c_uint32), ("front", C.c_uint32),
                ("t", C.c_float), ("p", C.c_float * 3), ("normal", C.c_float * 3), ("u", C.c_float), ("v", C.c_float),
                ("_pad", C.c_uint32)]


assert C.sizeof(vk_node) == 32 and C.sizeof(vk_sphere) == 16 and C.sizeof(vk_msphere) == 48
assert C.sizeof(vk_rect) == 32 and C.sizeof(vk_box) == 32 and C.sizeof(vk_xform) == 32
assert C.sizeof(vk_medium) == 16 and C.sizeof(vk_material) == 16 and C.sizeof(vk_texture) == 16
assert C.sizeof(vk_camera) == 96 and C.sizeof(vk_ray) == 36 and C.sizeof(vk_hit) == 56

# numpy views of the two batch structs (tests build ray batches with numpy)
import numpy as _np

RAY_DTYPE = _np.dtype([("origin", "<f4", 3), ("direction", "<f4", 3), ("time", "<f4"), ("tmin", "<f4"), ("tmax", "<f4")])
HIT_DTYPE = _np.dtype([("prim", "<u4"), ("face", "<u4"), ("mat", "<u4"), ("front", "<u4"), ("t", "<f4"),
                       ("p", "<f4", 3), ("normal", "<f4", 3), ("u", "<f4"), ("v", "<f4"), ("_pad", "<u4")])
# vk_eval (the shading-side parity hook): inputs, then results
EVAL_DTYPE = _np.dtype([("op", "<u4"), ("index", "<u4"), ("ray_o", "<f4", 3), ("ray_d", "<f4", 3), ("ray_time", "<f4"),
                        ("p", "<f4", 3), ("normal", "<f4", 3), ("t", "<f4"), ("u", "<f4"), ("v", "<f4"), ("front", "<u4"),
                        ("dir", "<f4", 3), ("xi", "<u4", 5),
                        ("alive", "<u4"), ("valid", "<u4"), ("out_o", "<f4", 3), ("out_d", "<f4", 3), ("out_time", "<f4"),
                        ("beta", "<f4", 3), ("L", "<f4", 3), ("value", "<f4")])
assert RAY_DTYPE.itemsize == 36 and HIT_DTYPE.itemsize == 56 and EVAL_DTYPE.itemsize == 43 * 4


class vk_adaptive_target(C.Structure):
    _fields_ = [("spp", C.c_uint32), ("min_spp", C.c_uint32), ("max_error", C.c_float)]
