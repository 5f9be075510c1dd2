"""vecchio_b200 -- B200-native (sm_100a) implementation of vecchio's path-tracing sample loop.

Python is only the harness language here (tests, bench).  The product is two shared libraries:

* ``lib/libvecchio_gpu.so``  -- hand-written CUDA kernels behind the C ABI of ``include/vecchio_gpu.h``
* ``lib/libvecchio_host.so`` -- the reference's scene/Hittable/Material API on the host with ``lower()``

There is no CPU fallback: :class:`Context` raises if the CUDA library is missing or no device exists.
"""
import ctypes as C
import os
import weakref

import numpy as np

from . import _abi
from ._abi import *  # noqa: F401,F403  (struct mirrors and constants)

_HERE = os.path.dirname(os.path.abspath(__file__))
REPO_ROOT = os.path.dirname(_HERE)
ASSETS_DIR = os.path.join(REPO_ROOT, "assets")
_LIBDIR = os.path.join(_HERE, "lib")

_host = None
_gpu = None


class VecchioError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[{code}] {msg}")
        self.code = code


def host_lib():
    """libvecchio_host.so (scene front end); built by `make host`."""
    global _host
    if _host is None:
        path = os.path.join(_LIBDIR, "libvecchio_host.so")
        if not os.path.exists(path):
            raise ImportError(f"{path} is missing: run `make host` (or __graft_entry__.build())")
        L = C.CDLL(path)
        L.vkh_scene_build.argtypes = [C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint32, C.POINTER(C.c_void_p)]
        L.vkh_scene_build.restype = C.c_int
        L.vkh_scene_free.argtypes = [C.c_void_p]
        L.vkh_scene_free.restype = None
        L.vkh_scene_desc.argtypes = [C.c_void_p]
        L.vkh_scene_desc.restype = C.POINTER(_abi.vk_scene_desc)
        L.vkh_scene_aspect_ratio.argtypes = [C.c_void_p]
        L.vkh_scene_aspect_ratio.restype = C.c_float
        L.vkh_scene_next_camera.argtypes = [C.c_void_p, C.POINTER(_abi.vk_camera)]
        L.vkh_scene_next_camera.restype = C.c_int
        L.vkh_camera_new.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_float,
                                     C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.POINTER(_abi.vk_camera)]
        L.vkh_camera_new.restype = None
        L.vkh_decode_png.argtypes = [C.c_char_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.vkh_decode_png.restype = C.c_long
        L.vkh_frame_to_rgb8.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
        L.vkh_frame_to_rgb8.restype = None
        L.vkh_write_ppm.argtypes = [C.c_char_p, C.c_void_p, C.c_uint32, C.c_uint32]
        L.vkh_write_ppm.restype = C.c_int
        L.vkh_write_pfm.argtypes = [C.c_char_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]
        L.vkh_write_pfm.restype = C.c_int
        L.vkh_frame_filename.argtypes = [C.c_char_p, C.c_uint32, C.c_char_p, C.c_size_t]
        L.vkh_frame_filename.restype = C.c_int
        L.vkh_last_error.restype = C.c_char_p
        _host = L
    return _host


def gpu_lib():
    """libvecchio_gpu.so (CUDA kernels + C ABI); built by `make gpu`.  Raises if absent."""
    global _gpu
    if _gpu is None:
        path = os.environ.get("VECCHIO_GPU_LIB") or os.path.join(_LIBDIR, "libvecchio_gpu.so")  # env: tuning sweeps
        if not os.path.exists(path):
            raise ImportError(f"{path} is missing: run `make gpu` (or __graft_entry__.build()). "
                              "There is no CPU fallback for the render path.")
        L = C.CDLL(path)
        vp = C.c_void_p
        L.vk_create.argtypes = [C.c_int, C.POINTER(vp)]
        L.vk_destroy.argtypes = [vp]
        L.vk_destroy.restype = None
        L.vk_last_error.argtypes = [vp]
        L.vk_last_error.restype = C.c_char_p
        L.vk_scene_upload.argtypes = [vp, C.POINTER(_abi.vk_scene_desc)]
        L.vk_render.argtypes = [vp, C.POINTER(_abi.vk_camera), C.POINTER(_abi.vk_render_params), vp, vp,
                                C.POINTER(_abi.vk_stats)]
        L.vk_scene_check.argtypes = [C.POINTER(_abi.vk_scene_desc), C.POINTER(_abi.vk_scene_info), C.c_char_p, C.c_size_t]
        L.vk_scene_check.restype = C.c_int
        L.vk_render_rgb8.argtypes = [vp, C.POINTER(_abi.vk_camera), C.POINTER(_abi.vk_render_params), vp, C.POINTER(_abi.vk_stats)]
        L.vk_render_device.argtypes = [vp, C.POINTER(_abi.vk_camera), C.POINTER(_abi.vk_render_params), vp, vp,
                                       C.POINTER(_abi.vk_stats)]
        L.vk_finalize_device.argtypes = [vp, vp, vp, C.c_size_t, C.c_uint32]
        L.vk_set_stream.argtypes = [vp, vp]
        L.vk_flush_stats.argtypes = [vp, C.POINTER(_abi.vk_stats)]
        L.vk_intersect.argtypes = [vp, vp, C.c_size_t, vp, C.c_uint32, vp]
        L.vk_eval_batch.argtypes = [vp, vp, C.c_size_t, C.c_uint32]
        L.vk_measure_peaks.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
        L.vk_device_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_char_p, C.c_size_t]
        L.vk_multi_create.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]
        L.vk_multi_destroy.argtypes = [vp]
        L.vk_multi_destroy.restype = None
        L.vk_multi_last_error.argtypes = [vp]
        L.vk_multi_last_error.restype = C.c_char_p
        L.vk_multi_device_count.argtypes = [vp]
        L.vk_multi_scene_upload.argtypes = [vp, C.POINTER(_abi.vk_scene_desc)]
        L.vk_multi_render.argtypes = [vp, C.POINTER(_abi.vk_camera), C.POINTER(_abi.vk_render_params), vp, vp, C.POINTER(_abi.vk_stats)]
        L.vk_multi_render_rgb8.argtypes = [vp, C.POINTER(_abi.vk_camera), C.POINTER(_abi.vk_render_params), vp, C.POINTER(_abi.vk_stats)]
        L.vk_render_frames.argtypes = [vp, C.POINTER(_abi.vk_camera), C.c_uint32, C.POINTER(_abi.vk_render_params), vp, C.POINTER(_abi.vk_stats)]
        L.vk_render_frames_rgb8.argtypes = [vp, C.POINTER(_abi.vk_camera), C.c_uint32, C.POINTER(_abi.vk_render_params), vp,
                                            C.POINTER(_abi.vk_stats)]
        L.vk_multi_render_frames_rgb8.argtypes = [vp, C.POINTER(_abi.vk_camera), C.c_uint32, C.POINTER(_abi.vk_render_params), vp,
                                                  C.POINTER(_abi.vk_stats)]
        L.vk_render_aov.argtypes = [vp, C.POINTER(_abi.vk_camera), C.c_uint32, C.POINTER(_abi.vk_render_params), C.c_uint32, vp, vp, vp, vp,
                                    C.POINTER(_abi.vk_stats)]
        L.vk_multi_render_aov.argtypes = L.vk_render_aov.argtypes
        L.vk_render_adaptive.argtypes = [vp, C.POINTER(_abi.vk_camera), C.POINTER(_abi.vk_render_params), C.c_uint32, C.c_float, vp, vp,
                                         C.POINTER(_abi.vk_stats)]
        L.vk_render_adaptive_rgb8.argtypes = [vp, C.POINTER(_abi.vk_camera), C.POINTER(_abi.vk_render_params), C.c_uint32, C.c_float, vp,
                                              vp, C.POINTER(_abi.vk_stats)]
        L.vk_render_frames_adaptive.argtypes = [vp, C.POINTER(_abi.vk_camera), C.c_uint32, C.POINTER(_abi.vk_render_params), C.c_uint32,
                                                C.c_float, vp, vp, C.POINTER(_abi.vk_stats)]
        L.vk_render_frames_adaptive_rgb8.argtypes = [vp, C.POINTER(_abi.vk_camera), C.c_uint32, C.POINTER(_abi.vk_render_params), C.c_uint32,
                                                     C.c_float, vp, vp, C.POINTER(_abi.vk_stats)]
        L.vk_adaptive_begin.argtypes = [vp, C.POINTER(_abi.vk_camera), C.c_uint32, C.POINTER(_abi.vk_render_params), C.c_uint32,
                                        C.POINTER(vp)]
        L.vk_adaptive_refine.argtypes = [vp, C.POINTER(_abi.vk_adaptive_target), C.POINTER(_abi.vk_stats)]
        L.vk_adaptive_read.argtypes = [vp, vp, vp, vp]
        L.vk_adaptive_read_rgb8.argtypes = [vp, vp, vp, vp]
        L.vk_adaptive_export.argtypes = [vp, vp, vp, vp, C.POINTER(_abi.vk_adaptive_target)]
        L.vk_adaptive_import.argtypes = [vp, vp, vp, vp, C.POINTER(_abi.vk_adaptive_target)]
        L.vk_adaptive_variant.argtypes = [vp]
        L.vk_adaptive_variant.restype = C.c_uint32
        L.vk_adaptive_destroy.argtypes = [vp]
        L.vk_adaptive_destroy.restype = None
        L.vk_adaptive_begin_shard.argtypes = [vp, C.POINTER(_abi.vk_camera), C.c_uint32, C.POINTER(_abi.vk_render_params), C.c_uint32,
                                              C.c_uint32, C.c_uint32, C.POINTER(vp)]
        for f in ("begin", "refine", "read", "read_rgb8", "export", "import", "variant", "destroy"):  # the same arguments over a vk_multi
            getattr(L, "vk_multi_adaptive_" + f).argtypes = getattr(L, "vk_adaptive_" + f).argtypes
            getattr(L, "vk_multi_adaptive_" + f).restype = getattr(L, "vk_adaptive_" + f).restype
        L.vk_multi_render_adaptive_rgb8.argtypes = L.vk_render_adaptive_rgb8.argtypes
        L.vk_multi_render_frames_adaptive_rgb8.argtypes = L.vk_render_frames_adaptive_rgb8.argtypes
        for f in ("vk_multi_create", "vk_multi_device_count", "vk_multi_scene_upload", "vk_multi_render", "vk_multi_render_rgb8",
                  "vk_multi_render_frames_rgb8", "vk_multi_render_adaptive_rgb8", "vk_multi_render_frames_adaptive_rgb8",
                  "vk_adaptive_begin_shard", "vk_multi_render_aov"):
            getattr(L, f).restype = C.c_int
        for f in ("vk_create", "vk_scene_upload", "vk_render", "vk_render_rgb8", "vk_render_device", "vk_finalize_device",
                  "vk_set_stream", "vk_flush_stats", "vk_intersect", "vk_eval_batch", "vk_measure_peaks", "vk_device_info",
                  "vk_render_frames", "vk_render_frames_rgb8", "vk_render_adaptive", "vk_render_adaptive_rgb8",
                  "vk_render_frames_adaptive", "vk_render_frames_adaptive_rgb8", "vk_adaptive_begin", "vk_adaptive_refine",
                  "vk_adaptive_read", "vk_adaptive_read_rgb8", "vk_adaptive_export", "vk_adaptive_import", "vk_render_aov"):
            getattr(L, f).restype = C.c_int
        _gpu = L
    return _gpu


GPU_SYMBOLS = ["vk_create", "vk_destroy", "vk_last_error", "vk_scene_check", "vk_scene_upload", "vk_render", "vk_render_rgb8", "vk_render_device",
               "vk_finalize_device", "vk_set_stream", "vk_flush_stats", "vk_intersect", "vk_eval_batch", "vk_measure_peaks",
               "vk_device_info", "vk_multi_create", "vk_multi_destroy", "vk_multi_last_error", "vk_multi_device_count",
               "vk_multi_scene_upload", "vk_multi_render", "vk_multi_render_rgb8", "vk_render_frames", "vk_render_frames_rgb8",
               "vk_multi_render_frames_rgb8", "vk_render_adaptive", "vk_render_adaptive_rgb8", "vk_render_frames_adaptive",
               "vk_render_frames_adaptive_rgb8", "vk_adaptive_begin", "vk_adaptive_refine", "vk_adaptive_read", "vk_adaptive_read_rgb8",
               "vk_adaptive_export", "vk_adaptive_import", "vk_adaptive_variant", "vk_adaptive_destroy", "vk_adaptive_begin_shard",
               "vk_multi_adaptive_begin", "vk_multi_adaptive_refine", "vk_multi_adaptive_read", "vk_multi_adaptive_read_rgb8",
               "vk_multi_adaptive_export", "vk_multi_adaptive_import", "vk_multi_adaptive_variant", "vk_multi_adaptive_destroy",
               "vk_multi_render_adaptive_rgb8", "vk_multi_render_frames_adaptive_rgb8", "vk_render_aov", "vk_multi_render_aov"]
HOST_SYMBOLS = ["vkh_scene_build", "vkh_scene_free", "vkh_scene_desc", "vkh_scene_aspect_ratio",
                "vkh_scene_next_camera", "vkh_camera_new", "vkh_decode_png", "vkh_frame_to_rgb8", "vkh_write_ppm",
                "vkh_frame_filename", "vkh_last_error", "vkh_write_pfm"]


class Scene:
    """A scene built with the reference's scene API (src/scene.rs) and lowered for the GPU.

    ``Scene("cornell_box")`` mirrors ``cornell_box()`` + ``BVHNode::new(&mut config.world)``
    (src/main.rs:159-169).  ``seed`` stands in for the reference's unseeded thread_rng().
    """

    def __init__(self, name, seed=1, param=0, assets_dir=None):
        L = host_lib()
        h = C.c_void_p()
        rc = L.vkh_scene_build(name.encode(), seed, (assets_dir or ASSETS_DIR).encode(), param, C.byref(h))
        if rc != 0:
            raise VecchioError(rc, L.vkh_last_error().decode())
        self._h = h
        self.name = name
        self.desc_ptr = L.vkh_scene_desc(h)
        self.desc = self.desc_ptr.contents
        self.aspect_ratio = float(L.vkh_scene_aspect_ratio(h))

    def next_camera(self):
        """``config.cam_iter.next()`` (src/main.rs:176); None when exhausted."""
        cam = _abi.vk_camera()
        return cam if host_lib().vkh_scene_next_camera(self._h, C.byref(cam)) else None

    def height_for(self, width):
        """``((width as f32) / config.aspect_ratio) as usize`` (src/main.rs:172)."""
        return int(np.float32(width) / np.float32(self.aspect_ratio))

    def census(self):
        d = self.desc
        return {k: int(getattr(d, "n_" + k)) for k in
                ("nodes", "spheres", "mspheres", "rects", "boxes", "xforms", "media", "lights", "materials",
                 "textures", "perlins")} | {"texel_bytes": int(d.n_texel_bytes)}

    def nbytes(self):
        d = self.desc
        return (d.n_nodes * 32 + d.n_spheres * 20 + d.n_mspheres * 48 + d.n_rects * 32 + d.n_boxes * 32 +
                d.n_xforms * 32 + d.n_media * 16 + d.n_lights * 4 + d.n_materials * 16 + d.n_textures * 16 +
                int(d.n_texel_bytes) + d.n_perlins * C.sizeof(_abi.vk_perlin))

    def close(self):
        if getattr(self, "_h", None):
            host_lib().vkh_scene_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def scene_check(desc_ptr):
    """``vk_scene_check``: validate + plan the device layout on the host (no GPU needed).  Returns a dict of
    what ``vk_scene_upload`` would build; raises VecchioError exactly where the upload would fail."""
    info = _abi.vk_scene_info()
    err = C.create_string_buffer(256)
    rc = gpu_lib().vk_scene_check(desc_ptr, C.byref(info), err, 256)
    if rc != 0:
        raise VecchioError(rc, err.value.decode())
    return {n: int(getattr(info, n)) for n, _ in info._fields_}


def camera_new(lookfrom, lookat, vup, vfov, aspect_ratio, aperture, focus_dist, time0, time1):
    """``Camera::new`` (src/main.rs:71-109)."""
    f3 = lambda v: (C.c_float * 3)(*[float(x) for x in v])  # noqa: E731
    cam = _abi.vk_camera()
    host_lib().vkh_camera_new(f3(lookfrom), f3(lookat), f3(vup), vfov, aspect_ratio, aperture, focus_dist, time0,
                              time1, C.byref(cam))
    return cam


def decode_png(path):
    """``ImageTexture::new`` (src/material.rs:269-279): (h, w, 3) uint8."""
    L = host_lib()
    w, h = C.c_uint32(), C.c_uint32()
    n = L.vkh_decode_png(path.encode(), None, 0, C.byref(w), C.byref(h))
    if n < 0:
        raise VecchioError(-1, L.vkh_last_error().decode())
    buf = np.empty(n, dtype=np.uint8)
    L.vkh_decode_png(path.encode(), buf.ctypes.data, n, C.byref(w), C.byref(h))
    return buf.reshape(h.value, w.value, 3)


def frame_to_rgb8(frame):
    """``vkh_frame_to_rgb8``: an (H, W, 3) linear frame with row 0 = bottom (what ``Context.render`` returns) ->
    the (H, W, 3) uint8 numbers of the reference's P3 file, top row first (src/main.rs:209-212)."""
    frame = np.ascontiguousarray(frame, dtype=np.float32)
    h, w, _ = frame.shape
    out = np.empty((h, w, 3), dtype=np.uint8)
    host_lib().vkh_frame_to_rgb8(frame.ctypes.data, w, h, out.ctypes.data)
    return out


def frame_filename(file_idx, out_dir=""):
    """``format!("output_{:04}.ppm", file_idx)`` (src/main.rs:201), under out_dir."""
    buf = C.create_string_buffer(4096)
    if host_lib().vkh_frame_filename(out_dir.encode(), file_idx, buf, 4096) < 0:
        raise ValueError("frame file name too long")
    return buf.value.decode()


def write_ppm(path, rgb8):
    """``vkh_write_ppm``: the P3 writer of src/main.rs:201-213; rgb8 = (H, W, 3) uint8 in file order (what
    ``Context.render_rgb8`` and ``frame_to_rgb8`` return)."""
    rgb8 = np.ascontiguousarray(rgb8, dtype=np.uint8)
    h, w, _ = rgb8.shape
    L = host_lib()
    if L.vkh_write_ppm(path.encode(), rgb8.ctypes.data, w, h) != 0:
        raise VecchioError(-1, L.vkh_last_error().decode())


def write_pfm(path, plane):
    """``vkh_write_pfm``: an (H, W, 3) or (H, W) float plane with row 0 = bottom (what render_aov returns) as a
    little-endian PFM file."""
    a = np.ascontiguousarray(plane, dtype=np.float32)
    if a.ndim not in (2, 3) or (a.ndim == 3 and a.shape[2] != 3):
        raise ValueError("write_pfm: an (H, W, 3) or (H, W) plane")
    L = host_lib()
    if L.vkh_write_pfm(os.fsencode(path), a.ctypes.data, a.shape[1], a.shape[0], 3 if a.ndim == 3 else 1) != 0:
        raise VecchioError(-1, L.vkh_last_error().decode())


def render_params(width, height, spp, max_depth=100, seed=1, spp_begin=0, spp_count=0, variant=0, flags=0,
                  background=(0.0, 0.0, 0.0)):
    p = _abi.vk_render_params()
    p.width, p.height, p.spp, p.spp_begin, p.spp_count, p.max_depth = width, height, spp, spp_begin, spp_count, max_depth
    p.seed = seed
    p.background[:] = background
    p.variant, p.flags = variant, flags
    return p


def _camera_array(cams):
    """A list of vk_camera as one contiguous C array (what vk_render_frames* take).  An empty list is rejected here,
    before the library is called."""
    cams = list(cams)
    if not cams:
        raise ValueError("render_frames: at least one camera")
    return (_abi.vk_camera * len(cams))(*cams), len(cams)


AOV_PLANES = (("albedo", 3), ("normal", 3), ("depth", 1), ("coverage", 1))


def _render_aov(fn, handle, check, cams, params, aov_spp):
    """``vk_render_aov`` / ``vk_multi_render_aov`` of the (non-empty) list ``cams`` into the four planes, each (K, H, W, c)
    with rows bottom-up, c = 1 squeezed.  Returns (planes, stats)."""
    arr, k = _camera_array(cams)
    n = k * params.width * params.height
    out = {name: np.empty(n * c, dtype=np.float32) for name, c in AOV_PLANES}
    st = _abi.vk_stats()
    check(fn(handle, arr, k, C.byref(params), int(aov_spp), *(out[name].ctypes.data for name, _ in AOV_PLANES), C.byref(st)))
    return {name: out[name].reshape((k, params.height, params.width, c) if c > 1 else (k, params.height, params.width))
            for name, c in AOV_PLANES}, st


def _check_adaptive(pass_spp, max_error):
    """What vk_render_adaptive* refuse of their two own arguments, refused here before the library is called."""
    if int(pass_spp) < 1:
        raise ValueError("render_adaptive: pass_spp must be >= 1")
    if not float(max_error) >= 0.0:  # (NaN fails the comparison)
        raise ValueError("render_adaptive: max_error must be >= 0 (and not NaN)")


ADAPTIVE_MAX_SPP = 65536  # the limit of the fixed-point sums of squares (include/vecchio_gpu.h)


def _adaptive_target(max_error, spp, min_spp):
    """A session target as (spp, min_spp, max_error), max_error as the library holds it (float32); bad values are
    refused here, before the library is called."""
    if int(spp) < 1:
        raise ValueError("adaptive target: spp must be >= 1")
    if int(min_spp) < 0:
        raise ValueError("adaptive target: min_spp must be >= 0")
    if not float(max_error) >= 0.0:  # (NaN fails the comparison)
        raise ValueError("adaptive target: max_error must be >= 0 (and not NaN)")
    return int(spp), int(min_spp), float(np.float32(max_error))


def _check_tightens(reached, target, limit, pass_spp):
    """What vk_adaptive_refine refuses of a target after ``reached`` (None: a fresh session), refused here first:
    the target must lie within the session's limit and tighten what was reached (include/vecchio_gpu.h)."""
    spp, min_spp, max_error = target
    if spp > limit:
        raise ValueError(f"adaptive target: spp {spp} exceeds the session's limit params.spp = {limit}")
    if reached is None:
        return
    r_spp, r_min, r_err = reached
    if (max_error != 0.0) if r_err == 0.0 else (max_error != 0.0 and max_error > r_err):
        raise ValueError(f"adaptive target: max_error {max_error} loosens {r_err} (0 is the tightest: after 0 only 0 may follow)")
    if min_spp < r_min:
        raise ValueError(f"adaptive target: min_spp {min_spp} is below the {r_min} already reached (it may only rise)")
    if spp < r_spp:
        raise ValueError(f"adaptive target: spp {spp} is below the {r_spp} already reached (it may only rise)")
    if spp > r_spp and r_spp % pass_spp:
        raise ValueError(f"adaptive target: spp may rise only from a cap on the pass grid; {r_spp} is not a multiple of pass_spp = {pass_spp}")


def _check_shard(shard):
    """``shard`` as (k, n) ints, or None; what vk_adaptive_begin_shard refuses, refused here first."""
    if shard is None:
        return None
    k, n = (int(x) for x in shard)
    if n < 1 or not 0 <= k < n:
        raise ValueError(f"adaptive_session: shard (k, n) needs 0 <= k < n, got ({k}, {n})")
    return k, n


class AdaptiveSession:
    """``vk_adaptive_begin`` .. ``vk_adaptive_destroy``: an adaptive render whose state outlives a call.  ``refine`` moves
    it to tighter targets, each step ending bit for bit where a fresh session refined once to that target would; a fresh
    session refined to ``(max_error, params.spp)`` is ``render_adaptive`` / ``render_frames_adaptive``.  One camera gives
    (H, W) shapes, a list of K cameras (K, H, W).  Made by ``Context.adaptive_session``; keeps its context alive.

    ``shard=(k, n)`` (``vk_adaptive_begin_shard``) renders only the pixels shard k of n owns (batch-wide pixel g belongs to
    shard (g // 32) % n); the others stay 0, and the n shards' exports add up to the unsharded export bit for bit.  Over a
    :class:`MultiContext` the same methods call ``vk_multi_adaptive_*``: device k runs shard k, and every result equals a
    one-GPU session's."""

    shard = None  # (k, n) of a shard session
    _api = "vk_adaptive_"  # the C calls: vk_adaptive_* on a Context, vk_multi_adaptive_* on a MultiContext

    def __init__(self, ctx, cams, params, pass_spp, shard=None):
        if int(pass_spp) < 1:
            raise ValueError("adaptive_session: pass_spp must be >= 1")
        shard = _check_shard(shard)
        self.single = isinstance(cams, _abi.vk_camera)
        cams = [cams] if self.single else list(cams)
        if not cams:
            raise ValueError("adaptive_session: at least one camera")
        arr, k = _camera_array(cams)
        self._h = None
        self._api = ctx._adaptive_api
        h = C.c_void_p()
        if shard is None:
            ctx._check(getattr(ctx._L, self._api + "begin")(ctx._h, arr, k, C.byref(params), int(pass_spp), C.byref(h)))
        else:
            ctx._check(ctx._L.vk_adaptive_begin_shard(ctx._h, arr, k, C.byref(params), int(pass_spp), shard[0], shard[1], C.byref(h)))
            self.shard = shard
        self._ctx, self._L, self._h = ctx, ctx._L, h
        ctx._sessions.add(self)
        self.cams = [_abi.vk_camera.from_buffer_copy(c) for c in cams]
        self.params = _abi.vk_render_params.from_buffer_copy(params)
        self.pass_spp, self.n_frames = int(pass_spp), k
        self.variant = int(self._fn("variant")(h))
        self.reached = None  # the last target reached, (spp, min_spp, max_error)

    def _fn(self, name):
        return getattr(self._L, self._api + name)

    def _check(self, rc):
        self._ctx._check(rc)

    def _shape(self):
        hw = (self.params.height, self.params.width)
        return hw if self.single else (self.n_frames,) + hw

    def target(self, max_error, spp=None, min_spp=0):
        """The target (spp, min_spp, max_error) refine would move to; spp None = the session's limit."""
        return _adaptive_target(max_error, self.params.spp if spp is None else spp, min_spp)

    def refine(self, max_error, spp=None, min_spp=0):
        """``vk_adaptive_refine``: render until every pixel meets the target; returns this refine's stats (paths =
        samples added).  A target that loosens the one reached, or bad values, raise ValueError before the library."""
        t = self.target(max_error, spp, min_spp)
        _check_tightens(self.reached, t, self.params.spp, self.pass_spp)
        T = _abi.vk_adaptive_target(*t)
        st = _abi.vk_stats()
        self._check(self._fn("refine")(self._h, C.byref(T), C.byref(st)))
        self.reached = t
        return st

    def _read(self, fn, dtype):
        shape = self._shape()
        n = int(np.prod(shape))
        img = np.empty(n * 3, dtype=dtype)
        cnt = np.empty(n, dtype=np.uint32)
        err = np.empty(n, dtype=np.float32)
        self._check(fn(self._h, img.ctypes.data, cnt.ctypes.data, err.ctypes.data))
        return img.reshape(shape + (3,)), cnt.reshape(shape), err.reshape(shape)

    def read(self):
        """``vk_adaptive_read``: (means float32 with row 0 = bottom, counts, error map) in ``render_adaptive``'s layout;
        the error map is the largest channel error the rule sees, +inf below two samples."""
        return self._read(self._fn("read"), np.float32)

    def read_rgb8(self):
        """``vk_adaptive_read_rgb8``: read()'s image through to_color with row 0 = top, counts and errors in that order."""
        return self._read(self._fn("read_rgb8"), np.uint8)

    def export(self):
        """``vk_adaptive_export``: (sums int64, squares uint64, both shape + (3,), counts uint32, reached), the raw
        fixed-point state in the accumulators' order (rows bottom-up)."""
        shape = self._shape()
        sums = np.empty(shape + (3,), dtype=np.int64)
        squares = np.empty(shape + (3,), dtype=np.uint64)
        counts = np.empty(shape, dtype=np.uint32)
        T = _abi.vk_adaptive_target()
        self._check(self._fn("export")(self._h, sums.ctypes.data, squares.ctypes.data, counts.ctypes.data, C.byref(T)))
        return sums, squares, counts, (None if T.spp == 0 else (int(T.spp), int(T.min_spp), float(T.max_error)))

    def import_(self, sums, squares, counts, reached):
        """``vk_adaptive_import``: replace the state by an exported one (``reached`` None: a state that reached no
        target).  The library refuses counts off the pass grid or above the cap reached."""
        shape = self._shape()
        sums = np.ascontiguousarray(sums, dtype=np.int64)
        squares = np.ascontiguousarray(squares, dtype=np.uint64)
        counts = np.ascontiguousarray(counts, dtype=np.uint32)
        if sums.shape != shape + (3,) or squares.shape != shape + (3,) or counts.shape != shape:
            raise ValueError(f"import_: the session's shape is {shape}, the state's {counts.shape}")
        r = (0, 0, 0.0) if reached is None else _adaptive_target(reached[2], reached[0], reached[1])
        T = _abi.vk_adaptive_target(*r)
        self._check(self._fn("import")(self._h, sums.ctypes.data, squares.ctypes.data, counts.ctypes.data, C.byref(T)))
        self.reached = None if reached is None else r

    def key(self, scene_name, scene_seed, scene_param=0):
        """The identity a checkpoint of this session carries (``adaptive_checkpoint.session_key``)."""
        from .adaptive_checkpoint import session_key
        return session_key(scene_name, scene_seed, self.cams, self.params, self.pass_spp, self.variant, scene_param, self.shard)

    def _own_key(self, key):
        """``key`` if it is this session's identity (its scene fields with the session's own cameras, params, pass_spp
        and kernel); ValueError otherwise, so that a state is never saved under, or loaded into, another session."""
        key = dict(key)
        own = self.key(key.get("scene"), key.get("scene_seed", 0), key.get("scene_param", 0))
        diff = sorted(k for k in set(own) | set(key) if own.get(k) != key.get(k))
        if diff:
            raise ValueError(f"the key is not this session's identity (differs in {', '.join(diff)})")
        return own

    def save(self, path, key):
        """The exported state and ``key`` (this session's identity, ``key()``) in one ``.npz``, written by
        write-and-rename."""
        from .adaptive_checkpoint import save_state
        save_state(path, self._own_key(key), *self.export())

    def load(self, path, key):
        """Imports a checkpoint written for ``key``.  ValueError, before the library is called, when ``key`` is not
        this session's own identity (other cameras, params, pass_spp or kernel) or the file's identity differs."""
        from .adaptive_checkpoint import load_state
        self.import_(*load_state(path, self._own_key(key)))

    def close(self):
        if getattr(self, "_h", None):
            self._fn("destroy")(self._h)
            self._h = None
            self._ctx._sessions.discard(self)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Context:
    """One GPU context (``vk_create``).  Fails loudly without the CUDA library or a device."""

    _adaptive_api = "vk_adaptive_"

    def __init__(self, device=0):
        L = gpu_lib()
        h = C.c_void_p()
        rc = L.vk_create(device, C.byref(h))
        if rc != 0:
            raise VecchioError(rc, (L.vk_last_error(None) or b"").decode())
        self._h = h
        self._L = L
        self.device = device
        self._sessions = weakref.WeakSet()

    def _check(self, rc):
        if rc != 0:
            raise VecchioError(rc, (self._L.vk_last_error(self._h) or b"").decode())

    def adaptive_session(self, cams, params, pass_spp, shard=None):
        """``vk_adaptive_begin``: an :class:`AdaptiveSession` over one camera ((H, W) shapes) or a list of K
        ((K, H, W)); frame f uses seed ``params.seed + f`` and ``params.spp`` is the session's limit.  ``shard=(k, n)``:
        ``vk_adaptive_begin_shard``, only the pixels shard k of n owns."""
        return AdaptiveSession(self, cams, params, pass_spp, shard)

    def upload(self, scene):
        self._check(self._L.vk_scene_upload(self._h, scene.desc_ptr))

    def render(self, cam, params, want_sumsq=False):
        """``vk_render``: the whole sample loop, host buffers in and out.  Returns (rgb, sumsq, stats)."""
        n = params.width * params.height * 3
        rgb = np.empty(n, dtype=np.float32)
        sq = np.empty(n, dtype=np.float32) if want_sumsq else None
        st = _abi.vk_stats()
        self._check(self._L.vk_render(self._h, C.byref(cam), C.byref(params), rgb.ctypes.data,
                                      sq.ctypes.data if want_sumsq else None, C.byref(st)))
        shape = (params.height, params.width, 3)
        return rgb.reshape(shape), (sq.reshape(shape) if want_sumsq else None), st

    def render_rgb8(self, cam, params):
        """``vk_render_rgb8``: the frame as the reference's PPM holds it -- (H, W, 3) uint8, row 0 = top,
        every channel through ``Vec3::to_color`` (src/main.rs:201-214).  Returns (rgb8, stats)."""
        out = np.empty(params.width * params.height * 3, dtype=np.uint8)
        st = _abi.vk_stats()
        self._check(self._L.vk_render_rgb8(self._h, C.byref(cam), C.byref(params), out.ctypes.data, C.byref(st)))
        return out.reshape(params.height, params.width, 3), st

    def render_frames(self, cams, params):
        """``vk_render_frames``: K cameras in one launch, frame f with seed ``params.seed + f``; frame f equals
        ``render(cams[f], params with seed + f)`` bit for bit on the same kernel: always with VK_FLAG_STRICT_MATH or an
        explicit variant; with AUTO in the render build a batch large enough to change kernel rounds differently.  Returns ((K, H, W, 3) float32, stats of the batch)."""
        arr, k = _camera_array(cams)
        out = np.empty(k * params.width * params.height * 3, dtype=np.float32)
        st = _abi.vk_stats()
        self._check(self._L.vk_render_frames(self._h, arr, k, C.byref(params), out.ctypes.data, C.byref(st)))
        return out.reshape(k, params.height, params.width, 3), st

    def render_frames_rgb8(self, cams, params):
        """``vk_render_frames_rgb8``: as render_frames, every frame as render_rgb8 returns it (rows top-down).
        Returns ((K, H, W, 3) uint8, stats of the batch)."""
        arr, k = _camera_array(cams)
        out = np.empty(k * params.width * params.height * 3, dtype=np.uint8)
        st = _abi.vk_stats()
        self._check(self._L.vk_render_frames_rgb8(self._h, arr, k, C.byref(params), out.ctypes.data, C.byref(st)))
        return out.reshape(k, params.height, params.width, 3), st

    def render_aov(self, cam, params, aov_spp):
        """``vk_render_aov`` of one camera: the first-hit feature planes of the camera rays ``render(cam, params)`` traces
        first for samples 0 .. aov_spp-1 (the header states each plane; the planes depend on the cameras, size, seed,
        background and the flags STRICT_MATH, FORCE_BVH and SKY_BACKGROUND only).  Returns ({"albedo": (H, W, 3),
        "normal": (H, W, 3), "depth": (H, W), "coverage": (H, W)} float32 with row 0 = bottom, stats)."""
        planes, st = self.render_frames_aov([cam], params, aov_spp)
        return {name: v[0] for name, v in planes.items()}, st

    def render_frames_aov(self, cams, params, aov_spp):
        """``vk_render_aov`` of K cameras in one launch, frame f with seed ``params.seed + f``: frame f equals
        ``render_aov(cams[f], params with seed + f)`` bit for bit.  Returns (the planes with (K, ...) shapes, stats)."""
        return _render_aov(self._L.vk_render_aov, self._h, self._check, cams, params, aov_spp)

    def render_adaptive(self, cam, params, pass_spp, max_error):
        """``vk_render_adaptive``: each pixel renders passes of ``pass_spp`` samples until its displayed noise (half the
        width of sqrt(mean +- standard error) in 8-bit steps) is <= ``max_error``, or until ``params.spp`` samples
        (the header states the rule).  A pixel that stopped at n samples equals ``render`` with spp = n on the same kernel,
        bit for bit; the stopping rule makes the frame slightly biased.  ``max_error = 0`` renders ``params.spp`` everywhere.
        Returns (rgb (H, W, 3) float32 with row 0 = bottom like ``render``, spp (H, W) uint32 in the same order, stats)."""
        _check_adaptive(pass_spp, max_error)
        n = params.width * params.height
        rgb = np.empty(n * 3, dtype=np.float32)
        spp = np.empty(n, dtype=np.uint32)
        st = _abi.vk_stats()
        self._check(self._L.vk_render_adaptive(self._h, C.byref(cam), C.byref(params), int(pass_spp), float(max_error),
                                               rgb.ctypes.data, spp.ctypes.data, C.byref(st)))
        return rgb.reshape(params.height, params.width, 3), spp.reshape(params.height, params.width), st

    def render_adaptive_rgb8(self, cam, params, pass_spp, max_error):
        """``vk_render_adaptive_rgb8``: render_adaptive's frame as ``render_rgb8`` returns one (row 0 = top).
        Returns (rgb8 (H, W, 3) uint8, spp (H, W) uint32 with row 0 = top, stats)."""
        _check_adaptive(pass_spp, max_error)
        n = params.width * params.height
        out = np.empty(n * 3, dtype=np.uint8)
        spp = np.empty(n, dtype=np.uint32)
        st = _abi.vk_stats()
        self._check(self._L.vk_render_adaptive_rgb8(self._h, C.byref(cam), C.byref(params), int(pass_spp), float(max_error),
                                                    out.ctypes.data, spp.ctypes.data, C.byref(st)))
        return out.reshape(params.height, params.width, 3), spp.reshape(params.height, params.width), st

    def render_frames_adaptive(self, cams, params, pass_spp, max_error):
        """``vk_render_frames_adaptive``: render_adaptive over K cameras, every pass one launch over the active pixels of
        all frames; frame f uses seed ``params.seed + f``.  Frame f's image and counts equal
        ``render_adaptive(cams[f], params with seed + f, pass_spp, max_error)`` bit for bit with VK_FLAG_STRICT_MATH; AUTO decides
        on the batch's pass-0 path count, and in the render build a batch kernel may round some pixels differently (the header).  Returns ((K, H, W, 3) float32 with row 0 = bottom,
        (K, H, W) uint32 counts in the same order, stats of the batch)."""
        _check_adaptive(pass_spp, max_error)
        arr, k = _camera_array(cams)
        n = k * params.width * params.height
        rgb = np.empty(n * 3, dtype=np.float32)
        spp = np.empty(n, dtype=np.uint32)
        st = _abi.vk_stats()
        self._check(self._L.vk_render_frames_adaptive(self._h, arr, k, C.byref(params), int(pass_spp), float(max_error),
                                                      rgb.ctypes.data, spp.ctypes.data, C.byref(st)))
        return rgb.reshape(k, params.height, params.width, 3), spp.reshape(k, params.height, params.width), st

    def render_frames_adaptive_rgb8(self, cams, params, pass_spp, max_error):
        """``vk_render_frames_adaptive_rgb8``: render_frames_adaptive's frames as ``render_adaptive_rgb8`` returns each
        (row 0 = top).  Returns ((K, H, W, 3) uint8, (K, H, W) uint32 counts with row 0 = top, stats of the batch)."""
        _check_adaptive(pass_spp, max_error)
        arr, k = _camera_array(cams)
        n = k * params.width * params.height
        out = np.empty(n * 3, dtype=np.uint8)
        spp = np.empty(n, dtype=np.uint32)
        st = _abi.vk_stats()
        self._check(self._L.vk_render_frames_adaptive_rgb8(self._h, arr, k, C.byref(params), int(pass_spp), float(max_error),
                                                           out.ctypes.data, spp.ctypes.data, C.byref(st)))
        return out.reshape(k, params.height, params.width, 3), spp.reshape(k, params.height, params.width), st

    def render_device(self, cam, params, d_sum_ptr, d_sumsq_ptr=None, want_stats=True):
        """``vk_render_device``: per-pixel SUMS of an spp slice into device memory.  With
        ``want_stats=False`` the call only enqueues work (collect counts with flush_stats())."""
        st = _abi.vk_stats() if want_stats else None
        self._check(self._L.vk_render_device(self._h, C.byref(cam), C.byref(params), d_sum_ptr, d_sumsq_ptr,
                                             C.byref(st) if want_stats else None))
        return st

    def set_stream(self, stream_ptr):
        self._check(self._L.vk_set_stream(self._h, stream_ptr))

    def flush_stats(self):
        st = _abi.vk_stats()
        self._check(self._L.vk_flush_stats(self._h, C.byref(st)))
        return st

    def finalize_device(self, d_sum_ptr, d_rgb_ptr, n_floats, spp):
        self._check(self._L.vk_finalize_device(self._h, d_sum_ptr, d_rgb_ptr, n_floats, spp))

    def intersect(self, rays, medium_xi=None, flags=0):
        """``vk_intersect``: rays is a numpy array of RAY_DTYPE; returns HIT_DTYPE array."""
        rays = np.ascontiguousarray(rays, dtype=_abi.RAY_DTYPE)
        out = np.zeros(len(rays), dtype=_abi.HIT_DTYPE)
        xi = None
        if medium_xi is not None:
            xi = np.ascontiguousarray(medium_xi, dtype=np.float32)
            assert xi.size == len(rays) * _abi.VK_MEDIUM_XI_SLOTS
        self._check(self._L.vk_intersect(self._h, rays.ctypes.data, len(rays), xi.ctypes.data if xi is not None else None,
                                         flags, out.ctypes.data))
        return out

    def eval_batch(self, recs, flags=0):
        """``vk_eval_batch``: recs is a numpy array of EVAL_DTYPE (inputs filled in); returns a copy with the results."""
        out = np.ascontiguousarray(recs, dtype=_abi.EVAL_DTYPE).copy()
        self._check(self._L.vk_eval_batch(self._h, out.ctypes.data, len(out), flags))
        return out

    def measure_peaks(self):
        a, b = C.c_float(), C.c_float()
        self._check(self._L.vk_measure_peaks(self._h, C.byref(a), C.byref(b)))
        return float(a.value), float(b.value)

    def device_info(self):
        sm, khz = C.c_int(), C.c_int()
        name = C.create_string_buffer(128)
        self._check(self._L.vk_device_info(self._h, C.byref(sm), C.byref(khz), name, 128))
        return {"sm_count": sm.value, "clock_khz": khz.value, "name": name.value.decode()}

    def close(self):
        if getattr(self, "_h", None):
            for s in list(getattr(self, "_sessions", ())):  # (sessions borrow the context: they go first)
                s.close()
            self._L.vk_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiContext:
    """``vk_multi_create``: one context over several GPUs of the node (spp slices per device, the peers' integer
    accumulators added on the first device over NVLink).  Same frame as one GPU, bit for bit.  Adaptive sampling splits
    pixels instead: device k renders shard k of N (``adaptive_session``, ``render_adaptive_rgb8``), again the one-GPU
    result bit for bit."""

    _adaptive_api = "vk_multi_adaptive_"

    def __init__(self, devices):
        L = gpu_lib()
        h = C.c_void_p()
        arr = (C.c_int * len(devices))(*devices)
        rc = L.vk_multi_create(arr, len(devices), C.byref(h))
        if rc != 0:
            raise VecchioError(rc, (L.vk_multi_last_error(None) or b"").decode())
        self._h, self._L, self.devices = h, L, list(devices)
        self._sessions = weakref.WeakSet()

    def adaptive_session(self, cams, params, pass_spp):
        """``vk_multi_adaptive_begin``: :class:`AdaptiveSession`'s methods over all devices (device k renders the pixels
        shard k of N owns); image, counts, error map, export and paths equal ``Context.adaptive_session``'s, and its
        checkpoints are interchangeable with a one-GPU session's."""
        return AdaptiveSession(self, cams, params, pass_spp)

    def render_adaptive_rgb8(self, cam, params, pass_spp, max_error):
        """``vk_multi_render_adaptive_rgb8``: ``Context.render_adaptive_rgb8`` over all devices, the same bytes and counts.
        Returns (rgb8 (H, W, 3) uint8, spp (H, W) uint32 with row 0 = top, stats)."""
        _check_adaptive(pass_spp, max_error)
        n = params.width * params.height
        out = np.empty(n * 3, dtype=np.uint8)
        spp = np.empty(n, dtype=np.uint32)
        st = _abi.vk_stats()
        self._check(self._L.vk_multi_render_adaptive_rgb8(self._h, C.byref(cam), C.byref(params), int(pass_spp), float(max_error),
                                                          out.ctypes.data, spp.ctypes.data, C.byref(st)))
        return out.reshape(params.height, params.width, 3), spp.reshape(params.height, params.width), st

    def render_frames_adaptive_rgb8(self, cams, params, pass_spp, max_error):
        """``vk_multi_render_frames_adaptive_rgb8``: ``Context.render_frames_adaptive_rgb8`` over all devices, the same
        bytes and counts.  Returns ((K, H, W, 3) uint8, (K, H, W) uint32 counts with row 0 = top, stats of the batch)."""
        _check_adaptive(pass_spp, max_error)
        arr, k = _camera_array(cams)
        n = k * params.width * params.height
        out = np.empty(n * 3, dtype=np.uint8)
        spp = np.empty(n, dtype=np.uint32)
        st = _abi.vk_stats()
        self._check(self._L.vk_multi_render_frames_adaptive_rgb8(self._h, arr, k, C.byref(params), int(pass_spp), float(max_error),
                                                                 out.ctypes.data, spp.ctypes.data, C.byref(st)))
        return out.reshape(k, params.height, params.width, 3), spp.reshape(k, params.height, params.width), st

    def _check(self, rc):
        if rc != 0:
            raise VecchioError(rc, (self._L.vk_multi_last_error(self._h) or b"").decode())

    def upload(self, scene):
        self._check(self._L.vk_multi_scene_upload(self._h, scene.desc_ptr))

    def render(self, cam, params, want_sumsq=False):
        n = params.width * params.height * 3
        rgb = np.empty(n, dtype=np.float32)
        sq = np.empty(n, dtype=np.float32) if want_sumsq else None
        st = _abi.vk_stats()
        self._check(self._L.vk_multi_render(self._h, C.byref(cam), C.byref(params), rgb.ctypes.data,
                                            sq.ctypes.data if want_sumsq else None, C.byref(st)))
        shape = (params.height, params.width, 3)
        return rgb.reshape(shape), (sq.reshape(shape) if want_sumsq else None), st

    def render_rgb8(self, cam, params):
        out = np.empty(params.width * params.height * 3, dtype=np.uint8)
        st = _abi.vk_stats()
        self._check(self._L.vk_multi_render_rgb8(self._h, C.byref(cam), C.byref(params), out.ctypes.data, C.byref(st)))
        return out.reshape(params.height, params.width, 3), st

    def render_aov(self, cam, params, aov_spp):
        """``vk_multi_render_aov`` of one camera, on the first device (the one-GPU planes): the first-hit feature planes of the camera rays ``render(cam, params)`` traces
        first for samples 0 .. aov_spp-1 (the header states each plane; the planes depend on the cameras, size, seed,
        background and the flags STRICT_MATH, FORCE_BVH and SKY_BACKGROUND only).  Returns ({"albedo": (H, W, 3),
        "normal": (H, W, 3), "depth": (H, W), "coverage": (H, W)} float32 with row 0 = bottom, stats)."""
        planes, st = self.render_frames_aov([cam], params, aov_spp)
        return {name: v[0] for name, v in planes.items()}, st

    def render_frames_aov(self, cams, params, aov_spp):
        """``vk_multi_render_aov`` of K cameras in one launch, frame f with seed ``params.seed + f``: frame f equals
        ``render_aov(cams[f], params with seed + f)`` bit for bit.  Returns (the planes with (K, ...) shapes, stats)."""
        return _render_aov(self._L.vk_multi_render_aov, self._h, self._check, cams, params, aov_spp)

    def render_frames_rgb8(self, cams, params):
        """``vk_multi_render_frames_rgb8``: Context.render_frames_rgb8 over all devices, the same frames bit for bit as one GPU's batch."""
        arr, k = _camera_array(cams)
        out = np.empty(k * params.width * params.height * 3, dtype=np.uint8)
        st = _abi.vk_stats()
        self._check(self._L.vk_multi_render_frames_rgb8(self._h, arr, k, C.byref(params), out.ctypes.data, C.byref(st)))
        return out.reshape(k, params.height, params.width, 3), st

    def close(self):
        if getattr(self, "_h", None):
            for s in list(getattr(self, "_sessions", ())):  # (sessions borrow the devices: they go first)
                s.close()
            self._L.vk_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def to_color(rgb):
    """``Vec3::to_color`` (src/vec3.rs:54-61) on an (..., 3) float array -> uint8 (output only)."""
    with np.errstate(invalid="ignore"):
        s = np.sqrt(rgb.astype(np.float32))
        s = np.where(s < 0.0, 0.0, np.where(s > 0.999, 0.999, s))  # Vec3::clamp keeps NaN
        v = np.float32(256.0) * s.astype(np.float32)
        v = np.where(np.isnan(v), 0.0, v)  # `NaN as u32` == 0
    return v.astype(np.uint32).astype(np.uint8)
