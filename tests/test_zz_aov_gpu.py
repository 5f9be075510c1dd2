"""vk_render_aov on the GPU: the first-hit albedo, normal, depth and coverage of the render's own camera rays.

The strict build's planes equal a host model bit for bit: the camera rays rebuilt in numpy float32 (tests/aov_model.py),
traced by vk_intersect and shaded by vk_eval_batch's texture lookups, then the definition's tables in sample order.  The
same model over the oracle's hits and textures agrees within the hit-parity bars; the render build agrees with the strict
build up to silhouettes and ties; the rays are the render's (a depth-1 render lights exactly the pixels whose sample-0
ray hits the light's front); batches, errors, stats, the frame program's PFM files and several GPUs."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import aov_model as am
from conftest import ROOT, cuda_device_count, get_scene

pytestmark = pytest.mark.gpu
RENDER_BIN = os.path.join(ROOT, "vecchio_b200", "lib", "vecchio_gpu_render")
BACKGROUND = (0.2, 0.3, 0.5)
# the nine scenes of the hit-parity tests (scene, param)
SCENES = [("cornell_box", 0), ("cornell_smoke", 0), ("random_spheres_demo", 0), ("final_scene", 0), ("bowser_demo", 0),
          ("perlin_demo", 0), ("balls_demo", 0), ("stress_spheres", 64), ("api_surface_demo", 0)]
# (label, flags, background, sky): the planes of every mode against the model
MODES = [("flat", 0, (0.0, 0.0, 0.0), False), ("bvh", 2, (0.0, 0.0, 0.0), False), ("background", 0, BACKGROUND, False),
         ("sky", 8, (0.0, 0.0, 0.0), True)]


def view(vb, cam, aperture=0.0, focus=None, time0=None, time1=None):
    """cam's view (eye, direction, up, field of view, aspect) rebuilt by Camera::new with another lens and shutter."""
    f = lambda a: np.array(a[:], dtype=np.float64)  # noqa: E731
    o, llc, h, v, w = f(cam.origin), f(cam.lower_left_corner), f(cam.horizontal), f(cam.vertical), f(cam.w)
    dist = -np.dot(llc + h / 2 + v / 2 - o, w)  # the focus distance cam was built with
    vfov = np.degrees(2 * np.arctan(np.linalg.norm(v) / 2 / dist))
    return vb.camera_new(o, o - w, f(cam.v), vfov, np.linalg.norm(h) / np.linalg.norm(v), aperture,
                         dist if focus is None else focus, cam.time0 if time0 is None else time0,
                         cam.time1 if time1 is None else time1)


def model(vb, scene, cam, W, H, seed, n, trace, eval_batch, background=(0.0, 0.0, 0.0), sky=False, frame=0):
    """The host model's planes of n samples; trace(rays, xi) -> hits, eval_batch(records) -> records."""
    key = am.frame_key(seed, frame)
    samples = [am.camera_sample(cam, W, H, key, s) for s in range(n)]
    hits = [trace(r, xi) for r, xi in samples]
    return am.planes(samples, hits, am.materials_of(scene), eval_batch, W, H, background, sky)


def gpu_hooks(vb, ctx, flags):
    strict = vb.VK_FLAG_STRICT_MATH | (flags & vb.VK_FLAG_FORCE_BVH)
    return (lambda r, xi: ctx.intersect(r, xi, flags=strict)), (lambda recs: ctx.eval_batch(recs, flags=vb.VK_FLAG_STRICT_MATH))


def params(vb, W, H, seed=7, flags=0, background=(0.0, 0.0, 0.0), spp=4, depth=50):
    return vb.render_params(W, H, spp, depth, seed=seed, flags=flags, background=background)


def bit_equal(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def assert_planes_equal(got, want, label):
    for k in ("albedo", "normal", "depth", "coverage"):
        assert bit_equal(got[k], want[k]), (label, k, int((got[k].view(np.uint32) != want[k].view(np.uint32)).sum()))


def build_gap(a, b, tol):
    """How two sets of planes differ where rays may resolve differently (silhouettes, ties): the share of pixels whose
    coverage differs, and of the pixels where it agrees, the share with a relative depth or an absolute albedo / normal
    difference above tol; with the largest differences, for the log."""
    same = a["coverage"] == b["coverage"]
    hit = same & (a["coverage"] > 0)
    with np.errstate(invalid="ignore", divide="ignore"):
        rel = np.where(hit, np.abs(a["depth"] - b["depth"]) / np.abs(a["depth"]), 0.0)
    da, dn = np.abs(a["albedo"] - b["albedo"]).max(axis=-1), np.abs(a["normal"] - b["normal"]).max(axis=-1)
    off = same & ((rel > tol) | (da > tol) | (dn > tol))
    return {"coverage_differs": float((~same).mean()), "off": float(off.sum() / max(1, same.sum())),
            "depth_rel_max": float(rel[same].max()), "albedo_max": float(da[same].max()), "normal_max": float(dn[same].max())}


# ---------------------------------------------------------------------------------------------------------------------
# 1. Exact against the host model (strict build), every scene and mode, aov_spp 1 and 3
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,param", SCENES, ids=[s[0] for s in SCENES])
def test_strict_planes_equal_the_host_model_bit_for_bit(vb, ctx, name, param):
    scene, cam = get_scene(vb, name, param=param)
    ctx.upload(scene)
    W = 48
    H = scene.height_for(W)
    for label, flags, bg, sky in MODES:
        trace, ev = gpu_hooks(vb, ctx, flags)
        for n in (1, 3):
            want = model(vb, scene, cam, W, H, 7, n, trace, ev, bg, sky)
            got, st = ctx.render_aov(cam, params(vb, W, H, flags=flags | vb.VK_FLAG_STRICT_MATH, background=bg), n)
            assert_planes_equal(got, want, (name, label, n))
            assert st.paths == st.rays == W * H * n and st.launches == 1 and st.variant == 0
        print(name, label, "coverage", float(want["coverage"].mean()))


# ---------------------------------------------------------------------------------------------------------------------
# 2. The same model over the oracle's hits and textures
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,param", SCENES, ids=[s[0] for s in SCENES])
def test_strict_planes_agree_with_the_oracle(vb, po, ctx, name, param):
    scene, cam = get_scene(vb, name, param=param)
    ctx.upload(scene)
    o = po.OracleScene(scene)
    W = 48
    H = scene.height_for(W)
    want = model(vb, scene, cam, W, H, 7, 3, o.intersect, o.eval_batch, BACKGROUND)
    got, _ = ctx.render_aov(cam, params(vb, W, H, flags=vb.VK_FLAG_STRICT_MATH, background=BACKGROUND), 3)
    g = build_gap(got, want, 1e-5)
    print(name, g)
    # the bars of the oracle hit-parity tests: ids equal but for ties, t / normal / uv within 1e-5
    assert g["coverage_differs"] <= 5e-3 and g["off"] <= 1e-2, (name, g)


# ---------------------------------------------------------------------------------------------------------------------
# 3. The render build against the strict build
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,param", SCENES, ids=[s[0] for s in SCENES])
def test_render_build_planes_match_the_strict_build(vb, ctx, name, param):
    scene, cam = get_scene(vb, name, param=param)
    ctx.upload(scene)
    W = 160
    H = scene.height_for(W)
    a, _ = ctx.render_aov(cam, params(vb, W, H, flags=vb.VK_FLAG_STRICT_MATH, background=BACKGROUND), 4)
    b, _ = ctx.render_aov(cam, params(vb, W, H, flags=0, background=BACKGROUND), 4)
    g = build_gap(a, b, 1e-4)
    print(name, g)
    # Measured on a B200 (profiles/aov_gpu_tests_b200.log): coverage never differs, and the flat scenes stay within 1e-4
    # everywhere; on the BVH scenes of small spheres (random_spheres_demo, stress_spheres, final_scene) the two builds'
    # rounding of the camera ray and of the sphere test moves the hit point on spheres a few hundred pixels across by up
    # to ~1e-3 of their radius, and a sample near the edge between two spheres may land on the other one: up to 9 % of
    # the pixels there
    assert g["coverage_differs"] <= 5e-3 and g["off"] <= 0.12, (name, g)


# ---------------------------------------------------------------------------------------------------------------------
# 4. Thin lens and shutter (final_scene: moving spheres and media)
# ---------------------------------------------------------------------------------------------------------------------
def test_shutter_planes_equal_the_host_model(vb, ctx):
    scene, cam0 = get_scene(vb, "final_scene")
    ctx.upload(scene)
    cam = view(vb, cam0, time0=0.25, time1=0.5)
    W = 64
    H = scene.height_for(W)
    trace, ev = gpu_hooks(vb, ctx, 0)
    want = model(vb, scene, cam, W, H, 7, 3, trace, ev)
    got, _ = ctx.render_aov(cam, params(vb, W, H, flags=vb.VK_FLAG_STRICT_MATH), 3)
    assert_planes_equal(got, want, "shutter")


def test_thin_lens_planes_match_the_host_model(vb, ctx):
    scene, cam0 = get_scene(vb, "final_scene")
    ctx.upload(scene)
    cam = view(vb, cam0, aperture=20.0, focus=500.0, time0=0.25, time1=0.5)
    W = 96
    H = scene.height_for(W)
    trace, ev = gpu_hooks(vb, ctx, 0)
    want = model(vb, scene, cam, W, H, 7, 4, trace, ev)
    got, _ = ctx.render_aov(cam, params(vb, W, H, flags=vb.VK_FLAG_STRICT_MATH), 4)
    g = build_gap(got, want, 1e-4)
    print("thin lens", g)
    # (measured: 1.3 % of the pixels, where a sample's lens offset from __sincosf moves it across an edge)
    assert g["coverage_differs"] <= 5e-3 and g["off"] <= 0.03, g


# ---------------------------------------------------------------------------------------------------------------------
# 5. These are the render's rays
# ---------------------------------------------------------------------------------------------------------------------
def turntable(vb, k):
    s = vb.Scene("cornell_box")
    base = s.next_camera()
    cams = [base]
    for f in range(1, k):  # Camera::new with the eye moved sideways, same view direction
        eye = [base.origin[i] + 40.0 * f * base.u[i] for i in range(3)]
        cams.append(vb.camera_new(eye, [eye[i] - base.w[i] for i in range(3)], list(base.v), 40.0, 1.0, 0.0, 10.0,
                                  base.time0, base.time1))
    return s, cams


def test_depth_one_render_lights_the_pixels_whose_first_ray_hits_the_light(vb, ctx):
    s, cams = turntable(vb, 3)
    ctx.upload(s)
    W = H = 64
    mt = am.materials_of(s)[0]
    p = params(vb, W, H, seed=5, flags=vb.VK_FLAG_STRICT_MATH, spp=1, depth=1)
    frames, _ = ctx.render_frames(cams, p)
    planes, _ = ctx.render_frames_aov(cams, p, 1)
    for f, cam in enumerate(cams):
        rays, xi = am.camera_sample(cam, W, H, am.frame_key(5, f), 0)
        h = ctx.intersect(rays, xi, flags=vb.VK_FLAG_STRICT_MATH)
        light = ((h["prim"] != 0) & (mt[h["mat"]] == am.VK_M_DIFFUSE_LIGHT) & (h["front"] != 0)).reshape(H, W)
        lit = (frames[f] != 0).any(axis=-1)
        assert light.any() and np.array_equal(lit, light), (f, int(light.sum()), int(lit.sum()))
        assert (planes["albedo"][f][light] == 1.0).all() and (planes["coverage"][f][light] == 1.0).all(), f
    single, _, _ = ctx.render(cams[0], p)
    assert np.array_equal(single, frames[0])


# ---------------------------------------------------------------------------------------------------------------------
# 6. Batches
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("flags", [0, 1], ids=["render_build", "strict"])
@pytest.mark.parametrize("k", [1, 3])
def test_batch_frames_equal_single_calls(vb, ctx, flags, k):
    scene, cam0 = get_scene(vb, "random_spheres_demo")
    ctx.upload(scene)
    cams = [view(vb, cam0, time0=0.1 * f, time1=0.1 * f + 0.5) for f in range(k)]
    W, H = 37, 23
    p = params(vb, W, H, seed=2**32 - 2, flags=flags)
    batch, st = ctx.render_frames_aov(cams, p, 3)
    assert st.paths == st.rays == k * W * H * 3
    for f in range(k):
        one, _ = ctx.render_aov(cams[f], params(vb, W, H, seed=2**32 - 2 + f, flags=flags), 3)
        for name in one:
            assert bit_equal(batch[name][f], one[name]), (f, name)


def test_planes_ignore_spp_depth_variant_and_legacy(vb, ctx):
    scene, cam = get_scene(vb, "cornell_box")
    ctx.upload(scene)
    a, _ = ctx.render_aov(cam, vb.render_params(40, 40, 8, 50, seed=3), 2)
    b, _ = ctx.render_aov(cam, vb.render_params(40, 40, 1000, 1, seed=3, spp_begin=10, spp_count=5, variant=vb.VK_VARIANT_STAGED,
                                                flags=vb.VK_FLAG_LEGACY_SCATTER), 2)
    for k in a:
        assert bit_equal(a[k], b[k]), k


# ---------------------------------------------------------------------------------------------------------------------
# 7. Errors and stats
# ---------------------------------------------------------------------------------------------------------------------
def raw_call(vb, ctx, cams, p, aov_spp, outs):
    arr = (vb.vk_camera * max(1, len(cams)))(*cams)
    st = vb.vk_stats()
    ptrs = [o.ctypes.data if o is not None else None for o in outs]
    return ctx._L.vk_render_aov(ctx._h, arr, len(cams), p, aov_spp, *ptrs, st), st


def test_refusals_write_nothing(vb, ctx):
    scene, cam = get_scene(vb, "cornell_box")
    ctx.upload(scene)
    W, H = 16, 16
    sentinel = np.float32(-7.0)
    outs = [np.full(W * H * c, sentinel, dtype=np.float32) for c in (3, 3, 1, 1)]
    bad_time = view(vb, cam, time0=1.0, time1=1.0)
    good = params(vb, W, H)
    for label, cams, p, n, o in [("aov_spp 0", [cam], good, 0, outs), ("aov_spp 65537", [cam], good, 65537, outs),
                                 ("all null", [cam], good, 2, [None] * 4), ("no frames", [], good, 2, outs),
                                 ("time0 >= time1", [bad_time], good, 2, outs), ("max_depth 0", [cam], params(vb, W, H, depth=0), 2, outs)]:
        rc, _ = raw_call(vb, ctx, cams, p, n, o)
        assert rc == vb.VK_ERR_INVALID, label
        assert all((x == sentinel).all() for x in outs), label
    fresh = vb.Context(0)
    try:
        rc, _ = raw_call(vb, fresh, [cam], good, 2, outs)
        assert rc == vb.VK_ERR_NO_SCENE
    finally:
        fresh.close()
    rc, st = raw_call(vb, ctx, [cam], good, 65536, outs)  # the largest aov_spp
    assert rc == 0 and st.rays == W * H * 65536


def test_one_null_plane_still_fills_the_others(vb, ctx):
    scene, cam = get_scene(vb, "cornell_smoke")
    ctx.upload(scene)
    W, H = 24, 20
    full, _ = ctx.render_aov(cam, params(vb, W, H), 2)
    names = [n for n, _ in vb.AOV_PLANES]
    for skip in range(4):
        outs = [np.empty(W * H * c, dtype=np.float32) if i != skip else None for i, (_, c) in enumerate(vb.AOV_PLANES)]
        rc, st = raw_call(vb, ctx, [cam], params(vb, W, H), 2, outs)
        assert rc == 0 and st.paths == st.rays == W * H * 2
        for i, o in enumerate(outs):
            if o is not None:
                assert bit_equal(o.reshape(full[names[i]].shape), full[names[i]]), (skip, names[i])


# ---------------------------------------------------------------------------------------------------------------------
# 8. The frame program and several GPUs
# ---------------------------------------------------------------------------------------------------------------------
def read_pfm(path):
    with open(path, "rb") as f:
        kind = f.readline().strip()
        w, h = map(int, f.readline().split())
        scale = float(f.readline())
        data = np.frombuffer(f.read(), dtype="<f4" if scale < 0 else ">f4")
    return data.reshape(h, w, 3) if kind == b"PF" else data.reshape(h, w)


@pytest.mark.parametrize("batch", [1, 2])
def test_program_writes_the_planes_as_pfm(vb, ctx, batch):
    scene = vb.Scene("cornell_box")
    cam = scene.next_camera()
    W = 64
    H = scene.height_for(W)
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([RENDER_BIN, "--scene", "cornell_box", "--width", str(W), "--spp", "4", "--aov", "2", "--frames", "2",
                            "--batch", str(batch), "--seed", "9", "--out-dir", d, "--quiet"], capture_output=True, text=True, cwd=ROOT)
        assert r.returncode == 0, r.stderr
        ctx.upload(scene)
        f = 0
        while os.path.exists(os.path.join(d, f"output_{f:04d}.ppm")):
            want, _ = ctx.render_aov(cam if f == 0 else scene.next_camera(), params(vb, W, H, seed=9 + f), 2)
            for name in ("albedo", "normal", "depth"):
                assert bit_equal(read_pfm(os.path.join(d, f"{name}_{f:04d}.pfm")).astype(np.float32), want[name]), (f, name)
            f += 1
        assert f >= 1


@pytest.mark.skipif(cuda_device_count() < 2, reason="needs two GPUs")
def test_multi_gpu_planes_equal_one_gpu(vb, ctx):
    scene, cam = get_scene(vb, "final_scene")
    ctx.upload(scene)
    m = vb.MultiContext([0, 1])
    try:
        m.upload(scene)
        for flags in (0, vb.VK_FLAG_STRICT_MATH):
            p = params(vb, 50, 50, flags=flags)
            a, _ = ctx.render_aov(cam, p, 3)
            b, st = m.render_aov(cam, p, 3)
            assert st.rays == 50 * 50 * 3
            for k in a:
                assert bit_equal(a[k], b[k]), k
            fa, _ = ctx.render_frames_aov([cam, cam], p, 2)
            fb, _ = m.render_frames_aov([cam, cam], p, 2)
            for k in fa:
                assert bit_equal(fa[k], fb[k]), k
    finally:
        m.close()
