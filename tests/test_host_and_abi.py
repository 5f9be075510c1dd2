"""CPU tests of the host front end and of the C-ABI libraries (no compute on a GPU)."""
import ctypes as C
import hashlib
import os
import re

import numpy as np
import pytest

from conftest import HAS_GPU, ROOT, get_scene


def test_gpu_library_exports_every_declared_symbol(vb):
    hdr = open(os.path.join(ROOT, "include", "vecchio_gpu.h")).read()
    declared = set(re.findall(r"\b(vk_[a-z0-9_]+)\s*\(", hdr)) - {"vk_ctx"}
    assert declared == set(vb.GPU_SYMBOLS)
    lib = C.CDLL(os.path.join(ROOT, "vecchio_b200", "lib", "libvecchio_gpu.so"))
    for name in declared | {"vk_selftest_philox"}:
        assert hasattr(lib, name), name


def test_host_library_exports_every_declared_symbol(vb):
    hdr = open(os.path.join(ROOT, "include", "vecchio_host.h")).read()
    declared = set(re.findall(r"\b(vkh_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(vb.HOST_SYMBOLS)
    lib = vb.host_lib()
    for name in declared:
        assert hasattr(lib, name), name


@pytest.mark.skipif(HAS_GPU, reason="a GPU is present")
def test_no_cpu_fallback_without_a_device(vb):
    with pytest.raises(vb.VecchioError) as e:
        vb.Context(0)
    assert e.value.code == vb.VK_ERR_NO_DEVICE


def test_unknown_scene_is_an_error(vb):
    with pytest.raises(vb.VecchioError):
        vb.Scene("not_a_scene")


# SURVEY App. C: decoded RGB8 bytes of the texture assets (sha256 prefix, first texel, centre texel)
PNG_KAT = {
    "earthmap.png": ((512, 1024), "0651e147c9164cf9a7bb9c32", (255, 255, 255), (0, 2, 53)),
    "bowser_face.png": ((32, 44), "1e8dc13edbc59d9c1d9670ce", (88, 118, 131), (88, 118, 131)),
    "bowser_top.png": ((32, 44), "b5e8a89a67dcf11f8f3463cb", None, None),
    "bowser_back.png": ((32, 44), "153364d7b24ef0235d9eebcb", None, None),
    "bowser_side.png": ((32, 32), "171691359437ce950d0b80d0", (88, 118, 131), (0, 0, 0)),
    "twitter.png": ((1740, 2904), "a6a0a39b8891b7c27d589c37", None, None),
}


@pytest.mark.parametrize("name", sorted(PNG_KAT))
def test_png_decoder_matches_known_hashes(vb, name):
    shape, sha, first, centre = PNG_KAT[name]
    img = vb.decode_png(os.path.join(vb.ASSETS_DIR, name))
    assert img.shape == shape + (3,)
    assert hashlib.sha256(img.tobytes()).hexdigest().startswith(sha)
    if first:
        assert tuple(img[0, 0]) == first
        assert tuple(img[shape[0] // 2, shape[1] // 2]) == centre


def test_png_decoder_matches_pil(vb):
    Image = pytest.importorskip("PIL.Image")
    for name in ("earthmap.png", "bowser_face.png"):
        ref = np.asarray(Image.open(os.path.join(vb.ASSETS_DIR, name)).convert("RGB"))
        assert np.array_equal(ref, vb.decode_png(os.path.join(vb.ASSETS_DIR, name)))


def test_camera_new_cornell(vb):
    """Camera::new for the Cornell box (src/main.rs:71-109, src/scene.rs:708-728), SURVEY App. C."""
    _, cam = get_scene(vb, "cornell_box")
    assert np.allclose(list(cam.w), [0, 0, -1]) and np.allclose(list(cam.u), [-1, 0, 0]) and np.allclose(list(cam.v), [0, 1, 0])
    assert np.allclose(list(cam.horizontal), [-7.2794046, 0, 0], rtol=1e-6)
    assert np.allclose(list(cam.vertical), [0, 7.2794046, 0], rtol=1e-6)
    assert np.allclose(list(cam.lower_left_corner), [281.63970, 274.36030, -790.0], rtol=1e-6)
    assert cam.lens_radius == 0.0 and (cam.time0, cam.time1) == (0.0, 1.0)


def test_rotating_camera_first_frame(vb):
    """RotatingCamera first frame of random_spheres_demo (src/scene.rs:65-91, 254-281)."""
    s, cam = get_scene(vb, "random_spheres_demo")
    assert np.allclose(list(cam.origin), [18.126156, 2.5, 8.452366], rtol=1e-6)
    assert s.height_for(400) == 225 and s.height_for(900) == 506 and s.height_for(3840) == 2160


def bvh_nodes(n):  # f(1)=f(2)=1, f(n)=1+f(n//2)+f(n-n//2)  (src/accel.rs:102-135)
    return 1 if n <= 2 else 1 + bvh_nodes(n // 2) + bvh_nodes(n - n // 2)


def test_scene_census_matches_reference_builders(vb):
    c = get_scene(vb, "cornell_box")[0].census()
    # 8 top-level objects -> 7 nodes; 5 walls + light(flipped) + light(unflipped, light list) rects
    assert (c["nodes"], c["spheres"], c["rects"], c["boxes"], c["xforms"], c["lights"], c["materials"]) == (7, 1, 7, 1, 2, 1, 5)
    c = get_scene(vb, "cornell_smoke")[0].census()
    assert (c["nodes"], c["boxes"], c["xforms"], c["media"], c["materials"]) == (7, 2, 4, 2, 6)
    c = get_scene(vb, "final_scene")[0].census()
    assert c["nodes"] == bvh_nodes(11) + bvh_nodes(400) + bvh_nodes(1000) == 13 + 511 + 1023
    assert (c["spheres"], c["mspheres"], c["boxes"], c["media"], c["perlins"], c["texel_bytes"]) == (1006, 1, 400, 2, 1, 1572864)
    c = get_scene(vb, "random_spheres_demo")[0].census()
    n_top = c["spheres"] + 1  # + the flipped light rect
    assert c["nodes"] == bvh_nodes(n_top) and 470 <= c["spheres"] <= 488 and c["texel_bytes"] == 1572864
    c = get_scene(vb, "bowser_demo")[0].census()
    assert (c["boxes"], c["xforms"]) == (22, 4) and c["nodes"] == bvh_nodes(3) + bvh_nodes(28)


def test_bvh_structure_invariants(vb):
    """Every node's box encloses its children; single-object leaves have left == right."""
    s, _ = get_scene(vb, "final_scene")
    d = s.desc
    nodes = np.ctypeslib.as_array(C.cast(d.nodes, C.POINTER(C.c_uint32)), shape=(d.n_nodes, 8))
    f = nodes.view(np.float32)
    singles = 0
    for i in range(d.n_nodes):
        l, r = int(nodes[i, 3]), int(nodes[i, 7])
        singles += l == r
        for ch in (l, r):
            if vb.ref_type(ch) == vb.VK_T_NODE:
                j = vb.ref_index(ch)
                assert j > i  # depth-first numbering: children after parents
                assert np.all(f[j, 0:3] >= f[i, 0:3]) and np.all(f[j, 4:7] <= f[i, 4:7])
        if vb.ref_type(l) == vb.VK_T_NODE:
            assert vb.ref_index(l) == i + 1  # left subtree follows its parent immediately
    assert singles == 3 + 112 + 24  # n=11 -> 3, n=400 -> 112, n=1000 -> 24 (SURVEY App. B)


def test_scene_build_is_deterministic_per_seed(vb):
    a, b, c = vb.Scene("final_scene", seed=5), vb.Scene("final_scene", seed=5), vb.Scene("final_scene", seed=6)

    def sph(s):
        return np.ctypeslib.as_array(C.cast(s.desc.spheres, C.POINTER(C.c_float)), shape=(s.desc.n_spheres, 4)).copy()

    assert np.array_equal(sph(a), sph(b)) and not np.array_equal(sph(a), sph(c))


def test_stress_scene_small(vb):
    s = vb.Scene("stress_spheres", param=40)
    c = s.census()
    assert c["spheres"] == 1600 and c["nodes"] == bvh_nodes(1602) and c["lights"] == 1


# ---------------------------------------------------------------------------------------------------
# vk_scene_check: the validator and the device-layout planning of vk_scene_upload, without a device
# ---------------------------------------------------------------------------------------------------
def test_scene_check_plans_every_shipped_scene(vb):
    want = {  # scene: (flat program?, simple build?, dynamic megakernel?)
        "cornell_box": (True, True, False), "cornell_smoke": (True, True, False), "balls_demo": (True, False, False),
        "api_surface_demo": (True, False, False), "perlin_demo": (True, False, False), "random_spheres_demo": (False, False, False),
        "random_spheres_cover": (False, False, False), "final_scene": (False, False, False), "bowser_demo": (False, False, False),
        "book1_cover": (False, False, False), "furnace_demo": (True, True, False),
    }
    for name, (flat, simple, dyn) in want.items():
        s, _ = get_scene(vb, name)
        info = vb.scene_check(s.desc_ptr)
        whole = info["flat_entries"] > 0 and info["flat_subtrees"] == 0  # (a hybrid program keeps subtrees: still a BVH scene)
        assert (whole, bool(info["simple"]), bool(info["dynamic_megakernel"])) == (flat, simple, dyn), (name, info)
        assert info["stack_need"] <= 96 and info["wide_nodes"] >= 1
    c = vb.scene_check(get_scene(vb, "cornell_box")[0].desc_ptr)
    # 6 world rects (5 walls + the flipped light) + 6 box sides + 1 sphere, in the world frame + one instance frame
    assert (c["flat_entries"], c["flat_segments"]) == (13, 2)
    # render build: the Boxy once more as ONE slab-test entry; every rect and box side (Lambertian / light, no (u, v)) gets a
    # shading record the shade stage writes the HitRec from, the glass sphere does not
    assert (c["flat_boxes"], c["flat_direct"]) == (1, 12)
    sm = vb.scene_check(get_scene(vb, "cornell_smoke")[0].desc_ptr)
    assert (sm["flat_entries"], sm["flat_boxes"], sm["flat_direct"]) == (8, 0, 6)  # the two boxes are medium boundaries, not entries
    f = vb.scene_check(get_scene(vb, "final_scene")[0].desc_ptr)
    assert f["flat_subtrees"] == 2  # the hybrid program: what VK_VARIANT_WARPQ runs on this scene (AUTO keeps the lane megakernel)
    # 13 + 511 + 1023 binary nodes collapse into far fewer 4-wide nodes; two BVH levels (world, instanced spheres)
    assert f["wide_nodes"] < (13 + 511 + 1023) * 0.6 and f["wide_levels_instance"] >= 4


def test_hybrid_program_plan(vb, monkeypatch):
    """The mixed top of a heterogeneous scene as typed entries, its homogeneous subtrees as BVH entries; VECCHIO_HYBRID=0 turns it off."""
    f = vb.scene_check(get_scene(vb, "final_scene")[0].desc_ptr)
    # the 9 loose objects, plus the box field and the instanced sphere cluster as subtrees, in two frames
    assert (f["flat_entries"], f["flat_segments"], f["flat_subtrees"]) == (11, 2, 2)
    monkeypatch.setenv("VECCHIO_HYBRID", "0")
    f = vb.scene_check(get_scene(vb, "final_scene")[0].desc_ptr)
    assert (f["flat_entries"], f["flat_subtrees"]) == (0, 0)


def test_scene_check_big_bvh_selects_the_dynamic_megakernel(vb):
    s = vb.Scene("stress_spheres", param=260)  # 67 600 spheres -> 131 071 binary nodes
    info = vb.scene_check(s.desc_ptr)
    assert info["dynamic_megakernel"] == 1 and info["flat_entries"] == 0
    assert info["wide_nodes"] < 0.5 * s.desc.n_nodes and info["stack_need"] <= 96


def _broken(vb, name, mutate):
    """A private copy of a lowered scene with one field broken; returns the VecchioError code and message."""
    import copy
    s = vb.Scene(name)
    d = s.desc
    keep = mutate(d)  # may return objects that must stay alive
    try:
        vb.scene_check(s.desc_ptr)
    except vb.VecchioError as e:
        return e.code, str(e), keep
    return 0, "", keep


def test_scene_check_refuses_malformed_and_unsupported_scenes(vb):
    def bad_version(d): d.api_version = 99
    def bad_root(d): d.root = (vb.VK_T_NODE << 28) | 0x0FFFFFF
    def bad_material(d): d.sphere_mat[0] = 10_000
    def bad_texture_type(d): d.textures[0].type = 17
    def cycle(d): d.nodes[1].left = (vb.VK_T_NODE << 28) | 0  # node 1 points back at the root
    def nested_instance(d):  # the child of a Translate made an instance again -> a transform below a transform's BVH is refused
        d.xforms[1].child = d.root
    for mutate, code in ((bad_version, vb.VK_ERR_INVALID), (bad_root, vb.VK_ERR_INVALID), (bad_material, vb.VK_ERR_INVALID),
                         (bad_texture_type, vb.VK_ERR_INVALID), (cycle, vb.VK_ERR_INVALID)):
        rc, msg, _ = _broken(vb, "cornell_box", mutate)
        assert rc == code and msg, (mutate.__name__, rc, msg)
    rc, msg, _ = _broken(vb, "cornell_box", nested_instance)
    assert rc in (vb.VK_ERR_UNSUPPORTED, vb.VK_ERR_INVALID) and msg
    # an empty light list is a valid upload (only the legacy integrator can render it)
    assert vb.scene_check(get_scene(vb, "random_spheres_cover")[0].desc_ptr)["flat_entries"] == 0


# ---------------------------------------------------------------------------------------------------
# the headers are C, not C++: examples/minimal.c is built with a pedantic C11 compiler against both libraries
# ---------------------------------------------------------------------------------------------------
def build_minimal_c(tmp_path):
    import subprocess
    exe = str(tmp_path / "minimal")
    lib = os.path.join(ROOT, "vecchio_b200", "lib")
    r = subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I" + os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "examples", "minimal.c"), "-L" + lib, "-lvecchio_host", "-lvecchio_gpu",
                        "-Wl,-rpath," + lib, "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_c_abi_compiles_and_links_from_plain_c(tmp_path):
    import subprocess
    exe = build_minimal_c(tmp_path)
    r = subprocess.run([exe, str(tmp_path / "out.ppm")], capture_output=True, text=True, cwd=ROOT)
    assert "layout: 13 flat entries in 2 segments" in r.stderr  # vk_scene_check ran (host only)
    if not HAS_GPU:
        assert r.returncode == 1 and "no CPU fallback" in r.stderr and not (tmp_path / "out.ppm").exists()
