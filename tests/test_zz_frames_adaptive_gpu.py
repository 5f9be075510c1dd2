"""Adaptive sampling of a batch of frames on the GPU (vk_render_frames_adaptive, vk_render_frames_adaptive_rgb8): every pass
renders the active pixels of all K frames in one launch, and frame f's image and sample counts equal, bit for bit,
vk_render_adaptive(cams[f], seed + f) on the same kernel (a pixel's decision depends on its own integer sums only)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

_SCENES = {}


def scene_and_cams(vb, name, param=0, k=3):
    """k cameras: the scene's iterator while it turns, then Camera::new views moved sideways from the scene's own camera."""
    key = (name, param)
    if key not in _SCENES:
        s = vb.Scene(name, seed=1, param=param)
        cams = [s.next_camera()]
        while len(cams) < 4:
            c = s.next_camera()
            if c is None:
                break
            cams.append(c)
        base = cams[0]
        for f in range(len(cams), 4):
            eye = [base.origin[i] + 0.3 * f * base.u[i] for i in range(3)]
            cams.append(vb.camera_new(eye, [eye[i] - base.w[i] for i in range(3)], list(base.v), 40.0, 1.0, 0.0, 10.0,
                                      base.time0, base.time1))
        _SCENES[key] = (s, cams)
    s, cams = _SCENES[key]
    return s, cams[:k]


def params_like(vb, p, **kw):
    q = type(p).from_buffer_copy(p)
    for k, v in kw.items():
        setattr(q, k, v)
    return q


def median_error_target(vb, ctx, cam, p, pass_spp):
    """A max_error that stops about half the pixels after pass 0 (the header's rule from vk_render's sums at pass_spp)."""
    rgb, sq, _ = ctx.render(cam, params_like(vb, p, spp=pass_spp), want_sumsq=True)
    m = rgb.astype(np.float64)
    se = np.sqrt(np.maximum(sq.astype(np.float64) / pass_spp - m * m, 0.0) / (pass_spp - 1))
    e = (128.0 * (np.sqrt(np.maximum(m + se, 0.0)) - np.sqrt(np.maximum(m - se, 0.0)))).max(axis=-1)
    return max(float(np.median(e)), 0.01)


def single_frames(ctx, cams, p, pass_spp, max_error, rgb8=False):
    """vk_render_adaptive(_rgb8) of every camera with seed + f: (images, counts, stats)."""
    imgs, counts, stats = [], [], []
    for f, cam in enumerate(cams):
        q = type(p).from_buffer_copy(p)
        q.seed = p.seed + f
        img, n, st = (ctx.render_adaptive_rgb8 if rgb8 else ctx.render_adaptive)(cam, q, pass_spp, max_error)
        imgs.append(img)
        counts.append(n)
        stats.append(st)
    return np.stack(imgs), np.stack(counts), stats


# The render build's static lane megakernel for flat scenes lit by one rect (the VK_LIGHT0 flavour) rounds differently in its
# batch (FrameListArgs) and single-frame (ListArgs) instantiations: the compiler contracts multiply-adds per kernel.  There
# the strict build carries the bit-for-bit check, and the render build must give the same counts and almost every pixel.
ROUNDS_APART = {("cornell_box", "MEGAKERNEL"), ("api_surface_demo", "MEGAKERNEL")}


def check_batch(vb, ctx, name, param=0, k=3, width=64, height=None, spp=40, pass_spp=8, depth=30, seed=11, max_error=None,
                single_variant=None, rounds_apart=False, **kw):
    """The batch against its frames' single adaptive calls on the kernel the batch ran (or single_variant)."""
    scene, cams = scene_and_cams(vb, name, param, k)
    ctx.upload(scene)
    p = vb.render_params(width, height or scene.height_for(width), spp, depth, seed=seed, **kw)
    if max_error is None:
        max_error = median_error_target(vb, ctx, cams[0], p, pass_spp)
    rgb, n, st = ctx.render_frames_adaptive(cams, p, pass_spp, max_error)
    assert rgb.shape == (k, p.height, p.width, 3) and n.shape == (k, p.height, p.width)
    assert st.paths == int(n.sum(dtype=np.uint64))
    want, wn, sts = single_frames(ctx, cams, params_like(vb, p, variant=st.variant if single_variant is None else single_variant),
                                  pass_spp, max_error)
    for f in range(k):
        assert np.array_equal(n[f], wn[f]), (name, f, kw)
        if rounds_apart:
            same = np.all(rgb[f] == want[f], axis=-1).mean()
            assert same >= 0.9 and abs(rgb[f].mean() / want[f].mean() - 1.0) < 0.01, (name, f, kw, float(same))
        else:
            assert np.array_equal(rgb[f], want[f]), (name, f, kw)
    if single_variant is None and not rounds_apart:
        assert all(s.variant == st.variant for s in sts)
        assert st.rays == sum(s.rays for s in sts) and st.dropped_samples == sum(s.dropped_samples for s in sts)
    return rgb, n, st, max_error


SCENES = [("cornell_box", 0), ("cornell_smoke", 0), ("random_spheres_demo", 0), ("bowser_demo", 0), ("final_scene", 0),
          ("api_surface_demo", 0), ("stress_spheres", 300)]  # (300: a BVH the dynamic megakernel runs)


@pytest.mark.parametrize("strict", [False, True], ids=["render", "strict"])
@pytest.mark.parametrize("variant", ["WARPQ", "STEPQ", "MEGAKERNEL"])
@pytest.mark.parametrize("name,param", SCENES)
def test_batch_frames_equal_their_single_adaptive_renders(vb, ctx, name, param, variant, strict):
    _, n, _, _ = check_batch(vb, ctx, name, param, variant=getattr(vb, "VK_VARIANT_" + variant),
                             flags=vb.VK_FLAG_STRICT_MATH if strict else 0, rounds_apart=not strict and (name, variant) in ROUNDS_APART)
    assert len(np.unique(n)) >= 2, (name, np.unique(n))  # the target stops some pixels early and keeps others


@pytest.mark.parametrize("name,param", SCENES)
def test_batch_frames_equal_their_single_adaptive_renders_auto_strict(vb, ctx, name, param):
    check_batch(vb, ctx, name, param, flags=vb.VK_FLAG_STRICT_MATH)


@pytest.mark.parametrize("variant", ["WARPQ", "STEPQ", "MEGAKERNEL"])
@pytest.mark.parametrize("name,param", SCENES)
def test_ragged_frames(vb, ctx, name, param, variant):
    # 61 x 37 = 2257 pixels a frame: frame boundaries fall inside a warp-queue chunk and inside a lane-megakernel group
    # of 32 list entries; 45 = 5 passes of 8 and a short one of 5
    check_batch(vb, ctx, name, param, width=61, height=37, spp=45, variant=getattr(vb, "VK_VARIANT_" + variant),
                rounds_apart=(name, variant) in ROUNDS_APART)
    if (name, variant) in ROUNDS_APART:  # the same frames bit for bit with the reference's operation order
        check_batch(vb, ctx, name, param, width=61, height=37, spp=45, variant=getattr(vb, "VK_VARIANT_" + variant),
                    flags=vb.VK_FLAG_STRICT_MATH)


@pytest.mark.parametrize("variant", ["WARPQ", "STEPQ", "MEGAKERNEL"])
def test_a_frame_that_stops_after_pass_0_drops_out(vb, ctx, variant):
    scene, cams = scene_and_cams(vb, "random_spheres_demo", 0, 2)
    ctx.upload(scene)
    W, H = 64, scene.height_for(64)
    up = vb.camera_new([0.0, 5000.0, 0.0], [0.0, 6000.0, 0.0], [1.0, 0.0, 0.0], 20.0, W / H, 0.0, 10.0, cams[0].time0, cams[0].time1)
    batch = [cams[0], up, cams[1]]
    p = vb.render_params(W, H, 40, 30, seed=11, variant=getattr(vb, "VK_VARIANT_" + variant))
    black, _, _ = ctx.render(up, params_like(vb, p, spp=8, seed=12))
    assert not black.any()  # (the premise: this camera sees only the black background)
    e = median_error_target(vb, ctx, cams[0], p, 8)
    rgb, n, st = ctx.render_frames_adaptive(batch, p, 8, e)
    assert np.all(n[1] == 8) and not rgb[1].any()
    want, wn, _ = single_frames(ctx, batch, params_like(vb, p, variant=st.variant), 8, e)
    assert np.array_equal(n, wn) and np.array_equal(rgb, want)
    assert n[0].max() > 8 and n[2].max() > 8


@pytest.mark.parametrize("name,param", [("cornell_box", 0), ("random_spheres_demo", 0), ("stress_spheres", 300)])
def test_one_frame_is_render_adaptive(vb, ctx, name, param):
    scene, cams = scene_and_cams(vb, name, param, 1)
    ctx.upload(scene)
    p = vb.render_params(64, scene.height_for(64), 40, 30, seed=7)
    e = median_error_target(vb, ctx, cams[0], p, 8)
    rgb, n, st = ctx.render_frames_adaptive(cams, p, 8, e)
    want, wn, sw = ctx.render_adaptive(cams[0], p, 8, e)
    assert np.array_equal(rgb[0], want) and np.array_equal(n[0], wn)
    assert (st.paths, st.rays, st.variant) == (sw.paths, sw.rays, sw.variant)
    rgb8, n8, _ = ctx.render_frames_adaptive_rgb8(cams, p, 8, e)
    want8, wn8, _ = ctx.render_adaptive_rgb8(cams[0], p, 8, e)
    assert np.array_equal(rgb8[0], want8) and np.array_equal(n8[0], wn8)


@pytest.mark.parametrize("name,param", SCENES)
def test_max_error_zero_is_render_frames_at_the_cap(vb, ctx, name, param):
    scene, cams = scene_and_cams(vb, name, param, 3)
    ctx.upload(scene)
    p = vb.render_params(64, scene.height_for(64), 24, 30, seed=3)
    rgb, n, st = ctx.render_frames_adaptive(cams, p, 8, 0.0)
    want, sw = ctx.render_frames(cams, params_like(vb, p, variant=st.variant))
    assert np.all(n == 24) and np.array_equal(rgb, want)
    assert st.paths == sw.paths == n.size * 24 and st.rays == sw.rays
    rgb8, n8, st8 = ctx.render_frames_adaptive_rgb8(cams, p, 8, 0.0)
    want8, _ = ctx.render_frames_rgb8(cams, params_like(vb, p, variant=st8.variant))
    assert np.all(n8 == 24) and np.array_equal(rgb8, want8)


@pytest.mark.parametrize("name,param", [("cornell_box", 0), ("final_scene", 0), ("stress_spheres", 300)])
def test_huge_max_error_is_render_frames_at_pass_spp(vb, ctx, name, param):
    scene, cams = scene_and_cams(vb, name, param, 3)
    ctx.upload(scene)
    p = vb.render_params(64, scene.height_for(64), 64, 30, seed=3)
    rgb, n, st = ctx.render_frames_adaptive(cams, p, 8, 1e9)
    want, _ = ctx.render_frames(cams, params_like(vb, p, spp=8, variant=st.variant))
    assert np.all(n == 8) and np.array_equal(rgb, want) and st.paths == n.size * 8


@pytest.mark.parametrize("name,param", [("cornell_smoke", 0), ("random_spheres_demo", 0), ("final_scene", 0)])
def test_rgb8_frames_equal_render_adaptive_rgb8(vb, ctx, name, param):
    _, n, st, e = check_batch(vb, ctx, name, param, spp=48)
    scene, cams = scene_and_cams(vb, name, param, 3)
    p = vb.render_params(64, scene.height_for(64), 48, 30, seed=11)
    rgb8, n8, st8 = ctx.render_frames_adaptive_rgb8(cams, p, 8, e)
    assert st8.variant == st.variant and st8.paths == st.paths
    assert np.array_equal(n8, n[:, ::-1])  # the counts follow the image: each frame's top row first
    want, wn, _ = single_frames(ctx, cams, params_like(vb, p, variant=st8.variant), 8, e, rgb8=True)
    assert np.array_equal(rgb8, want) and np.array_equal(n8, wn)


def test_auto_decides_on_the_batch(vb, ctx):
    scene, cams = scene_and_cams(vb, "random_spheres_demo", 0, 2)
    ctx.upload(scene)
    # pass 0 of one 400 x 225 frame is 2.88 M paths (lane megakernel), of the pair 5.76 M (step queues)
    p = vb.render_params(400, 225, 64, 50, seed=1)
    e = median_error_target(vb, ctx, cams[0], p, 32)
    q = params_like(vb, p, flags=vb.VK_FLAG_STRICT_MATH)
    rgb, n, st = ctx.render_frames_adaptive(cams, q, 32, e)
    want, wn, sts = single_frames(ctx, cams, q, 32, e)
    assert st.variant == vb.VK_VARIANT_STEPQ and sts[0].variant == vb.VK_VARIANT_MEGAKERNEL
    assert np.array_equal(n, wn) and np.array_equal(rgb, want)  # the reference's operation order on both kernels
    # the render build contracts FMAs per kernel: there the frames equal single calls on the batch's kernel
    rgb, n, st = ctx.render_frames_adaptive(cams, p, 32, e)
    assert st.variant == vb.VK_VARIANT_STEPQ
    want, wn, _ = single_frames(ctx, cams, params_like(vb, p, variant=st.variant), 32, e)
    assert np.array_equal(n, wn) and np.array_equal(rgb, want)


def test_stats_and_determinism(vb, ctx):
    scene, cams = scene_and_cams(vb, "final_scene", 0, 3)
    ctx.upload(scene)
    p = vb.render_params(96, 96, 64, 50, seed=5)
    a = ctx.render_frames_adaptive(cams, p, 8, 6.0)
    b = ctx.render_frames_adaptive(cams, p, 8, 6.0)
    assert a[2].paths == int(a[1].sum(dtype=np.uint64)) and a[2].launches > 0 and a[2].ms_kernels > 0
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[0], b[0])
    assert (a[2].paths, a[2].rays, a[2].dropped_samples, a[2].variant) == (b[2].paths, b[2].rays, b[2].dropped_samples, b[2].variant)


def _raw(ctx, vb, cams, n, p, pass_spp=8, max_error=1.0, fn="vk_render_frames_adaptive", out=True):
    arr = (vb.vk_camera * max(len(cams), 1))(*cams) if cams else None
    img = np.empty(64 * 64 * 3 * 4, dtype=np.float32)
    cnt = np.empty(64 * 64 * 4, dtype=np.uint32)
    st = vb.vk_stats()
    rc = getattr(ctx._L, fn)(ctx._h, arr, n, C.byref(p) if p is not None else None, pass_spp, max_error,
                             img.ctypes.data if out else None, cnt.ctypes.data, C.byref(st))
    return rc, (ctx._L.vk_last_error(ctx._h) or b"").decode()


def test_errors(vb, ctx):
    scene, cams = scene_and_cams(vb, "random_spheres_demo", 0, 3)
    p = vb.render_params(32, 18, 16, 10, seed=1)
    fresh = vb.Context(0)
    rc, msg = _raw(fresh, vb, cams, 3, p)
    assert rc == vb.VK_ERR_NO_SCENE, msg
    fresh.close()
    ctx.upload(scene)
    for fn in ("vk_render_frames_adaptive", "vk_render_frames_adaptive_rgb8"):
        assert _raw(ctx, vb, cams, 0, p, fn=fn)[0] == vb.VK_ERR_INVALID
        assert _raw(ctx, vb, [], 3, p, fn=fn)[0] == vb.VK_ERR_INVALID
        assert _raw(ctx, vb, cams, 3, None, fn=fn)[0] == vb.VK_ERR_INVALID
        assert _raw(ctx, vb, cams, 3, p, fn=fn, out=False)[0] == vb.VK_ERR_INVALID
        assert _raw(ctx, vb, cams, 3, p, pass_spp=0, fn=fn)[0] == vb.VK_ERR_INVALID
        assert _raw(ctx, vb, cams, 3, p, max_error=-1.0, fn=fn)[0] == vb.VK_ERR_INVALID
        assert _raw(ctx, vb, cams, 3, p, max_error=float("nan"), fn=fn)[0] == vb.VK_ERR_INVALID
    assert _raw(ctx, vb, cams, 3, params_like(vb, p, spp_begin=1))[0] == vb.VK_ERR_INVALID
    assert _raw(ctx, vb, cams, 3, params_like(vb, p, spp_count=8))[0] == vb.VK_ERR_INVALID
    rc, msg = _raw(ctx, vb, cams, 3, params_like(vb, p, spp=65537))
    assert rc == vb.VK_ERR_INVALID and "65536" in msg, msg
    bad = [vb.vk_camera.from_buffer_copy(c) for c in cams]
    bad[2].time0, bad[2].time1 = 1.0, 1.0
    rc, msg = _raw(ctx, vb, bad, 3, p)
    assert rc == vb.VK_ERR_INVALID and "frame 2" in msg, msg
    big = vb.render_params(8192, 8192, 1, 10, seed=1)  # 8192^2 * 3 * 11 > 2^31 - 1: refused before anything is allocated
    rc, msg = _raw(ctx, vb, cams * 4, 11, big, pass_spp=1)
    assert rc == vb.VK_ERR_INVALID and "too large" in msg, msg
    for v in (vb.VK_VARIANT_STAGED, vb.VK_VARIANT_WAVEFRONT):
        assert _raw(ctx, vb, cams, 3, params_like(vb, p, variant=v))[0] == vb.VK_ERR_UNSUPPORTED
    # the context still renders after every refusal
    check_batch(vb, ctx, "random_spheres_demo")


SELFCHECK_LIB = os.path.join(ROOT, "build", "libvk_selfcheck.so")
SELFCHECK_CHILD = r"""
import ctypes as C, hashlib, sys
sys.path.insert(0, %r)
import numpy as np
import vecchio_b200 as vb
L = vb.gpu_lib()
L.vk_debug_counters.argtypes = [C.c_void_p, C.POINTER(C.c_ulonglong)]
ctx = vb.Context(0)
WQ, SQ = vb.VK_VARIANT_WARPQ, vb.VK_VARIANT_STEPQ
for name, W, variant in (("cornell_box", 61, WQ), ("cornell_smoke", 48, WQ), ("random_spheres_demo", 61, WQ),
                         ("random_spheres_demo", 61, SQ), ("final_scene", 48, SQ)):
    s = vb.Scene(name, seed=1); cams = [s.next_camera()]
    while len(cams) < 3:
        c = s.next_camera()
        cams.append(c if c is not None else cams[-1])
    ctx.upload(s)
    # (the self-check counter holds the last pass's violations: 1e9 stops every pixel after pass 0, 4 keeps some to the cap)
    for e in (1e9, 4.0):
        rgb, n, st = ctx.render_frames_adaptive(cams, vb.render_params(W, s.height_for(W), 40, 50, seed=3, variant=variant), 8, e)
        out = (C.c_ulonglong * 8)(); L.vk_debug_counters(ctx._h, out)
        print(name + ":" + str(variant), e, st.paths, st.rays, int(out[5]),
              hashlib.sha256(rgb.tobytes() + n.tobytes()).hexdigest()[:16], flush=True)
"""


def _run_selfcheck_child(lib):
    env = dict(os.environ)
    if lib:
        env["VECCHIO_GPU_LIB"] = lib
    r = subprocess.run([sys.executable, "-c", SELFCHECK_CHILD % ROOT], capture_output=True, text=True, env=env, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    return [line.split() for line in r.stdout.strip().splitlines()]


def test_queue_protocol_selfcheck_on_batched_adaptive_passes():
    if not os.path.exists(SELFCHECK_LIB):
        subprocess.run([os.path.join(ROOT, "scripts", "build_variants.sh"), "selfcheck:-DVKQ_SELFCHECK=1"], check=True, cwd=ROOT,
                       stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    checked, normal = _run_selfcheck_child(SELFCHECK_LIB), _run_selfcheck_child(None)
    assert len(checked) == len(normal) == 10
    for c, n in zip(checked, normal):
        assert int(c[4]) == 0, ("queue protocol violations", c)
        assert c[:4] == n[:4] and c[5] == n[5], ("the self-checking build renders other frames", c, n)
