"""Adaptive sampling on the GPU (vk_render_adaptive, vk_render_adaptive_rgb8, the program's --adaptive): a pixel that stopped
at n samples holds exactly its global samples [0, n), so its mean is vk_render(spp = n)'s pixel on the same kernel, bit for
bit; the stopping rule is the one the header states; the passes use the pass grid; errors come before any launch."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from test_frames_and_checkpoints import RENDER_BIN

pytestmark = pytest.mark.gpu

_SCENES = {}


def scene_and_cam(vb, name, param=0):
    key = (name, param)
    if key not in _SCENES:
        s = vb.Scene(name, seed=1, param=param)
        _SCENES[key] = (s, s.next_camera())
    return _SCENES[key]


def params_like(vb, p, **kw):
    q = type(p).from_buffer_copy(p)
    for k, v in kw.items():
        setattr(q, k, v)
    return q


def rule_error(rgb, sumsq, n):
    """The header's per-pixel error (largest channel) from vk_render's means and sums of squares at n samples."""
    m = rgb.astype(np.float64)
    se = np.sqrt(np.maximum(sumsq.astype(np.float64) / n - m * m, 0.0) / (n - 1))
    e = 128.0 * (np.sqrt(np.maximum(m + se, 0.0)) - np.sqrt(np.maximum(m - se, 0.0)))
    return e.max(axis=-1)


def median_error_target(vb, ctx, cam, p, pass_spp):
    """A max_error that stops about half the pixels after pass 0, so the frame ends with several sample counts."""
    rgb, sq, _ = ctx.render(cam, params_like(vb, p, spp=pass_spp), want_sumsq=True)
    return max(float(np.median(rule_error(rgb, sq, pass_spp))), 0.01)  # (> 0: a target of 0 never stops early)


def on_pass_grid(n, pass_spp, spp):
    return np.all((n == spp) | ((n % pass_spp == 0) & (n > 0) & (n <= spp)))


def check_prefix(vb, ctx, name, param=0, width=64, height=None, spp=40, pass_spp=8, depth=30, seed=11, max_error=None, **kw):
    scene, cam = scene_and_cam(vb, name, param)
    ctx.upload(scene)
    p = vb.render_params(width, height or scene.height_for(width), spp, depth, seed=seed, **kw)
    if max_error is None:
        max_error = median_error_target(vb, ctx, cam, p, pass_spp)
    rgb, n, st = ctx.render_adaptive(cam, p, pass_spp, max_error)
    assert on_pass_grid(n, pass_spp, spp), (name, np.unique(n))
    assert st.paths == int(n.sum(dtype=np.uint64)), (name, st.paths)
    # the fixed render at each count, on the kernel the adaptive call ran (AUTO decides on pass 0's path count there)
    q = params_like(vb, p, variant=st.variant)
    for v in np.unique(n):
        want, _, sw = ctx.render(cam, params_like(vb, q, spp=int(v)))
        assert sw.variant == st.variant
        sel = n == v
        assert np.array_equal(rgb[sel], want[sel]), (name, int(v), kw)
    return rgb, n, st, max_error


SCENES = [("cornell_box", 0), ("cornell_smoke", 0), ("random_spheres_demo", 0), ("bowser_demo", 0), ("final_scene", 0),
          ("api_surface_demo", 0), ("stress_spheres", 300)]  # (300: a BVH the dynamic megakernel runs)


@pytest.mark.parametrize("strict", [False, True], ids=["render", "strict"])
@pytest.mark.parametrize("variant", ["AUTO", "WARPQ", "STEPQ", "MEGAKERNEL"])
@pytest.mark.parametrize("name,param", SCENES)
def test_adaptive_pixels_equal_fixed_renders_at_their_count(vb, ctx, name, param, variant, strict):
    _, n, _, _ = check_prefix(vb, ctx, name, param, variant=getattr(vb, "VK_VARIANT_" + variant),
                              flags=vb.VK_FLAG_STRICT_MATH if strict else 0)
    assert len(np.unique(n)) >= 2, (name, np.unique(n))  # the target stops some pixels early and keeps others


@pytest.mark.parametrize("variant", ["AUTO", "WARPQ", "STEPQ", "MEGAKERNEL"])
def test_adaptive_legacy_sky(vb, ctx, variant):
    check_prefix(vb, ctx, "random_spheres_cover", variant=getattr(vb, "VK_VARIANT_" + variant),
                 flags=vb.VK_FLAG_LEGACY_SCATTER | vb.VK_FLAG_SKY_BACKGROUND)


@pytest.mark.parametrize("name,param", SCENES)
def test_adaptive_ragged_size(vb, ctx, name, param):
    # 61 x 37 = 2257 pixels: the warp queues' last list chunk and the lane megakernel's last group of 32 are partial;
    # 45 = 5 passes of 8 and a short one of 5
    check_prefix(vb, ctx, name, param, width=61, height=37, spp=45)


@pytest.mark.parametrize("name,param", [("cornell_box", 0), ("random_spheres_demo", 0), ("final_scene", 0), ("stress_spheres", 300)])
def test_adaptive_at_a_few_hundred_thousand_paths_per_pass(vb, ctx, name, param):
    check_prefix(vb, ctx, name, param, width=300, spp=32, pass_spp=8, depth=50)


@pytest.mark.parametrize("name,param", SCENES)
def test_max_error_zero_is_the_fixed_render(vb, ctx, name, param):
    scene, cam = scene_and_cam(vb, name, param)
    ctx.upload(scene)
    p = vb.render_params(64, scene.height_for(64), 24, 30, seed=3)
    rgb, n, st = ctx.render_adaptive(cam, p, 8, 0.0)
    want, _, sw = ctx.render(cam, params_like(vb, p, variant=st.variant))
    assert np.all(n == 24) and np.array_equal(rgb, want)
    assert st.paths == 64 * scene.height_for(64) * 24 and st.rays == sw.rays
    rgb8, n8, st8 = ctx.render_adaptive_rgb8(cam, p, 8, 0.0)
    want8, _ = ctx.render_rgb8(cam, params_like(vb, p, variant=st8.variant))
    assert np.all(n8 == 24) and np.array_equal(rgb8, want8)


@pytest.mark.parametrize("name,param", [("cornell_box", 0), ("final_scene", 0), ("stress_spheres", 300)])
def test_huge_max_error_stops_after_pass_0(vb, ctx, name, param):
    scene, cam = scene_and_cam(vb, name, param)
    ctx.upload(scene)
    p = vb.render_params(64, scene.height_for(64), 64, 30, seed=3)
    rgb, n, st = ctx.render_adaptive(cam, p, 8, 1e9)
    want, _, _ = ctx.render(cam, params_like(vb, p, spp=8, variant=st.variant))
    assert np.all(n == 8) and np.array_equal(rgb, want) and st.paths == n.size * 8


@pytest.mark.parametrize("name,param", [("cornell_smoke", 0), ("final_scene", 0)])
def test_rgb8_pixels_equal_render_rgb8_at_their_count(vb, ctx, name, param):
    _, n, st, e = check_prefix(vb, ctx, name, param, spp=48)
    scene, cam = scene_and_cam(vb, name, param)
    p = vb.render_params(64, scene.height_for(64), 48, 30, seed=11)
    rgb8, n8, st8 = ctx.render_adaptive_rgb8(cam, p, 8, e)
    assert np.array_equal(n8, n[::-1]) and st8.paths == st.paths  # the counts follow the image: top row first
    for v in np.unique(n8):
        want, _ = ctx.render_rgb8(cam, params_like(vb, p, spp=int(v), variant=st8.variant))
        assert np.array_equal(rgb8[n8 == v], want[n8 == v]), (name, int(v))


def test_adaptive_is_deterministic(vb, ctx):
    scene, cam = scene_and_cam(vb, "final_scene")
    ctx.upload(scene)
    p = vb.render_params(96, 96, 64, 50, seed=5)
    a = ctx.render_adaptive(cam, p, 8, 6.0)
    b = ctx.render_adaptive(cam, p, 8, 6.0)
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[0], b[0])
    assert (a[2].paths, a[2].rays, a[2].dropped_samples) == (b[2].paths, b[2].rays, b[2].dropped_samples)


@pytest.mark.parametrize("name", ["cornell_box", "final_scene"])
def test_stopping_rule_matches_the_header(vb, ctx, name):
    # recomputed from vk_render's means and (double, then fp32) sums of squares at each pass's count: the decision may
    # differ from the fixed-point squares' only for pixels within 1 % of the threshold
    M, spp = 8, 48
    rgb, n, st, e = check_prefix(vb, ctx, name, width=96, spp=spp, pass_spp=M)
    scene, cam = scene_and_cam(vb, name)
    p = vb.render_params(96, scene.height_for(96), spp, 30, seed=11, variant=st.variant)
    for k in range(1, spp // M):
        nk = k * M
        active = n >= nk
        r, sq, _ = ctx.render(cam, params_like(vb, p, spp=nk), want_sumsq=True)
        err = rule_error(r, sq, nk)[active]
        stopped = (n == nk)[active]
        disagree = stopped != (err <= e)
        assert np.all(np.abs(err[disagree] - e) <= 0.01 * e), (name, nk, int(disagree.sum()))
    if name == "cornell_box":  # the light seen directly: every sample is its emission, no variance, done after pass 0
        r, sq, _ = ctx.render(cam, params_like(vb, p, spp=spp), want_sumsq=True)
        r64 = r.astype(np.float64)
        emitter = np.all(r64 > 1.0, axis=-1) & np.all(np.abs(sq / spp - r64 * r64) <= 1e-6 * r64 * r64, axis=-1)
        assert emitter.sum() > 10 and np.all(n[emitter] == M)


def test_quality_against_a_4x_reference(vb, ctx):
    scene, cam = scene_and_cam(vb, "cornell_box")
    ctx.upload(scene)
    cap, e = 1000, 2.0
    p = vb.render_params(600, 600, cap, 50, seed=1)
    rgb, n, st = ctx.render_adaptive(cam, p, 64, e)
    ref, _, _ = ctx.render(cam, vb.render_params(600, 600, 4 * cap, 50, seed=987654321))
    assert abs(rgb.mean() / ref.mean() - 1.0) < 0.01
    stopped = n < cap
    assert stopped.any()
    d = 256.0 * np.abs(np.sqrt(np.maximum(rgb[stopped], 0)) - np.sqrt(np.maximum(ref[stopped], 0)))
    assert (d <= 3 * e).mean() >= 0.95, float((d <= 3 * e).mean())


def _raw(ctx, vb, p, pass_spp=8, max_error=1.0, cam=None, fn="vk_render_adaptive"):
    out = np.empty(64 * 64 * 3, dtype=np.float32)
    cnt = np.empty(64 * 64, dtype=np.uint32)
    st = vb.vk_stats()
    camp = C.byref(cam) if cam is not None else None
    rc = getattr(ctx._L, fn)(ctx._h, camp, C.byref(p) if p is not None else None, pass_spp, max_error, out.ctypes.data,
                             cnt.ctypes.data, C.byref(st))
    return rc, (ctx._L.vk_last_error(ctx._h) or b"").decode()


def test_adaptive_errors(vb, ctx):
    scene, cam = scene_and_cam(vb, "random_spheres_demo")
    fresh = vb.Context(0)
    p = vb.render_params(32, 18, 16, 10, seed=1)
    assert _raw(fresh, vb, p, cam=cam)[0] == vb.VK_ERR_NO_SCENE
    fresh.close()
    ctx.upload(scene)
    for fn in ("vk_render_adaptive", "vk_render_adaptive_rgb8"):
        assert _raw(ctx, vb, p, pass_spp=0, cam=cam, fn=fn)[0] == vb.VK_ERR_INVALID
        assert _raw(ctx, vb, p, max_error=-1.0, cam=cam, fn=fn)[0] == vb.VK_ERR_INVALID
        assert _raw(ctx, vb, p, max_error=float("nan"), cam=cam, fn=fn)[0] == vb.VK_ERR_INVALID
        assert _raw(ctx, vb, None, cam=cam, fn=fn)[0] == vb.VK_ERR_INVALID
        assert _raw(ctx, vb, p, cam=None, fn=fn)[0] == vb.VK_ERR_INVALID
    assert _raw(ctx, vb, params_like(vb, p, spp_begin=1), cam=cam)[0] == vb.VK_ERR_INVALID
    assert _raw(ctx, vb, params_like(vb, p, spp_count=8), cam=cam)[0] == vb.VK_ERR_INVALID
    assert _raw(ctx, vb, params_like(vb, p, spp_count=16), cam=cam)[0] == 0  # spp_count == spp is the whole range
    rc, msg = _raw(ctx, vb, params_like(vb, p, spp=65537), cam=cam)
    assert rc == vb.VK_ERR_INVALID and "65536" in msg, msg
    assert _raw(ctx, vb, params_like(vb, p, width=1), cam=cam)[0] == vb.VK_ERR_INVALID
    assert _raw(ctx, vb, params_like(vb, p, variant=99), cam=cam)[0] == vb.VK_ERR_INVALID
    bad = vb.vk_camera.from_buffer_copy(cam)
    bad.time0, bad.time1 = 1.0, 1.0
    assert _raw(ctx, vb, p, cam=bad)[0] == vb.VK_ERR_INVALID
    for v in (vb.VK_VARIANT_STAGED, vb.VK_VARIANT_WAVEFRONT):
        assert _raw(ctx, vb, params_like(vb, p, variant=v), cam=cam)[0] == vb.VK_ERR_UNSUPPORTED
    # the context still renders after every refusal
    check_prefix(vb, ctx, "random_spheres_demo")


def test_program_adaptive_zero_writes_the_fixed_files(tmp_path):
    # config 1's size (random spheres, 400 x 225, 16 spp), strict: --adaptive 0 renders every sample of every pixel
    args = ["--scene", 3, "--width", 400, "--spp", 16, "--depth", 50, "--frames", 2, "--strict", "--quiet"]
    outs = []
    for sub, extra in (("fixed", []), ("adaptive", ["--adaptive", 0, "--pass-spp", 4])):
        out = tmp_path / sub
        out.mkdir()
        r = subprocess.run([RENDER_BIN, "--out-dir", str(out)] + [str(a) for a in args + extra], capture_output=True,
                           text=True, cwd=ROOT, timeout=600)
        assert r.returncode == 0, r.stderr
        outs.append(out)
    names = sorted(os.listdir(outs[0]))
    assert len(names) == 2 and names == sorted(os.listdir(outs[1]))
    for name in names:
        assert (outs[0] / name).read_bytes() == (outs[1] / name).read_bytes(), name


def test_program_adaptive_writes_a_frame(tmp_path):
    r = subprocess.run([RENDER_BIN, "--out-dir", str(tmp_path), "--scene", "1", "--width", "200", "--spp", "256", "--frames", "1",
                        "--adaptive", "3", "--pass-spp", "32"], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr
    assert os.listdir(tmp_path) == ["output_0000.ppm"]
