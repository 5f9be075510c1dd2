"""Batches of frames on the GPU (vk_render_frames, vk_render_frames_rgb8, vk_multi_render_frames_rgb8, the program's
--batch): frame f of a batch is the single-frame render of cams[f] with seed + f on the same kernel, bit for bit (integer
accumulators, Philox keyed per frame); with VK_FLAG_STRICT_MATH whatever kernels run the two."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from test_frames_and_checkpoints import RENDER_BIN, parse_ppm

pytestmark = pytest.mark.gpu

_SCENES = {}


def scene_and_cams(vb, name, param=0, k=5):
    """k cameras: the scene's iterator while it turns, then Camera::new views around the scene's own camera."""
    key = (name, param)
    if key not in _SCENES:
        s = vb.Scene(name, seed=1, param=param)
        cams = [s.next_camera()]
        while len(cams) < 5:
            c = s.next_camera()
            if c is None:
                break
            cams.append(c)
        base = cams[0]
        for f in range(len(cams), 5):  # a fixed-camera scene: Camera::new with the eye moved sideways, same view direction
            eye = [base.origin[i] + 0.3 * f * base.u[i] for i in range(3)]
            c = vb.camera_new(eye, [eye[i] - base.w[i] for i in range(3)], list(base.v), 40.0, 1.0, 0.0, 10.0,
                              base.time0, base.time1)
            cams.append(c)
        _SCENES[key] = (s, cams)
    s, cams = _SCENES[key]
    return s, cams[:k]


def singles(ctx, cams, p):
    out, stats = [], []
    for f, cam in enumerate(cams):
        q = type(p).from_buffer_copy(p)
        q.seed = p.seed + f
        rgb, _, st = ctx.render(cam, q)
        out.append(rgb)
        stats.append(st)
    return np.stack(out), stats


def check_batch(vb, ctx, name, param=0, k=3, width=64, spp=8, depth=30, seed=11, **kw):
    scene, cams = scene_and_cams(vb, name, param, k)
    ctx.upload(scene)
    p = vb.render_params(width, kw.pop("height", None) or scene.height_for(width), spp, depth, seed=seed, **kw)
    got, st = ctx.render_frames(cams, p)
    want, sts = singles(ctx, cams, p)
    assert got.shape == want.shape and np.array_equal(got, want), (name, k, kw)
    assert st.paths == sum(s.paths for s in sts) and st.rays == sum(s.rays for s in sts)
    assert st.dropped_samples == sum(s.dropped_samples for s in sts)
    return got, st


SCENES = [("cornell_box", 0), ("cornell_smoke", 0), ("random_spheres_demo", 0), ("bowser_demo", 0), ("final_scene", 0),
          ("api_surface_demo", 0), ("stress_spheres", 300)]  # (300: a BVH the dynamic megakernel runs, test_batch_frames.py)


@pytest.mark.parametrize("strict", [False, True], ids=["render", "strict"])
@pytest.mark.parametrize("k", [1, 3, 5])
@pytest.mark.parametrize("name,param", SCENES)
def test_batch_equals_single_frames_auto(vb, ctx, name, param, k, strict):
    check_batch(vb, ctx, name, param, k=k, flags=vb.VK_FLAG_STRICT_MATH if strict else 0)


@pytest.mark.parametrize("strict", [False, True], ids=["render", "strict"])
@pytest.mark.parametrize("variant", ["WARPQ", "STEPQ", "MEGAKERNEL"])
@pytest.mark.parametrize("name,param", SCENES)
def test_batch_equals_single_frames_explicit_variant(vb, ctx, name, param, variant, strict):
    check_batch(vb, ctx, name, param, k=3, variant=getattr(vb, "VK_VARIANT_" + variant),
                flags=vb.VK_FLAG_STRICT_MATH if strict else 0)


@pytest.mark.parametrize("variant", ["AUTO", "WARPQ", "STEPQ", "MEGAKERNEL"])
def test_batch_legacy_sky(vb, ctx, variant):
    check_batch(vb, ctx, "random_spheres_cover", k=3, variant=getattr(vb, "VK_VARIANT_" + variant),
                flags=vb.VK_FLAG_LEGACY_SCATTER | vb.VK_FLAG_SKY_BACKGROUND)


@pytest.mark.parametrize("name,param", SCENES)
def test_batch_ragged_size(vb, ctx, name, param):
    check_batch(vb, ctx, name, param, k=3, width=61, height=37)


@pytest.mark.parametrize("variant", ["WARPQ", "STEPQ", "MEGAKERNEL"])
@pytest.mark.parametrize("name,param", [("cornell_box", 0), ("cornell_smoke", 0), ("random_spheres_demo", 0), ("final_scene", 0),
                                        ("stress_spheres", 300)])
def test_batch_equals_single_frames_at_a_few_hundred_thousand_paths_per_frame(vb, ctx, name, param, variant):
    # 300 wide: two warp-queue chunks per row, the second one partial; 8 spp: 0.36 - 0.72 M paths per frame, so the lane
    # megakernels' items and units and the queue chunks cross every frame boundary with the whole GPU busy
    check_batch(vb, ctx, name, param, k=5, width=300, spp=8, depth=50, variant=getattr(vb, "VK_VARIANT_" + variant))


@pytest.mark.parametrize("name,param", [("cornell_smoke", 0), ("random_spheres_demo", 0), ("final_scene", 0)])
def test_batch_sample_slice(vb, ctx, name, param):
    check_batch(vb, ctx, name, param, k=3, spp=40, spp_begin=7, spp_count=21)


@pytest.mark.parametrize("name,param", SCENES)
def test_batch_rgb8_equals_render_rgb8(vb, ctx, name, param):
    scene, cams = scene_and_cams(vb, name, param, 3)
    ctx.upload(scene)
    p = vb.render_params(72, scene.height_for(72), 8, 30, seed=5)
    got, _ = ctx.render_frames_rgb8(cams, p)
    for f, cam in enumerate(cams):
        q = vb.render_params(72, scene.height_for(72), 8, 30, seed=5 + f)
        want, _ = ctx.render_rgb8(cam, q)
        assert np.array_equal(got[f], want), (name, f)


def test_auto_moves_a_config1_turntable_batch_onto_the_step_queues(vb, ctx):
    scene, cams = scene_and_cams(vb, "random_spheres_demo", 0, 3)
    ctx.upload(scene)
    p = vb.render_params(400, 225, 16, 50, seed=1)
    _, st1 = ctx.render_frames(cams[:1], p)
    assert st1.variant == vb.VK_VARIANT_MEGAKERNEL  # 1.44 M paths
    got, st3 = ctx.render_frames(cams, p)
    assert st3.variant == vb.VK_VARIANT_STEPQ  # 4.32 M paths in the batch
    # the render build contracts FMAs per kernel: the batch equals single frames on the same kernel there ...
    want, sts = singles(ctx, cams, vb.render_params(400, 225, 16, 50, seed=1, variant=vb.VK_VARIANT_STEPQ))
    assert np.array_equal(got, want)
    assert (st3.paths, st3.rays) == (sum(s.paths for s in sts), sum(s.rays for s in sts))
    # ... and with the reference's operation order the AUTO batch equals the AUTO single frames (lane megakernel) too
    q = vb.render_params(400, 225, 16, 50, seed=1, flags=vb.VK_FLAG_STRICT_MATH)
    got, st3 = ctx.render_frames(cams, q)
    want, sts = singles(ctx, cams, q)
    assert st3.variant == vb.VK_VARIANT_STEPQ and sts[0].variant == vb.VK_VARIANT_MEGAKERNEL
    assert np.array_equal(got, want) and st3.rays == sum(s.rays for s in sts)


def _raw(ctx, vb, cams, n, p, out=None, fn="vk_render_frames"):
    arr = (vb.vk_camera * max(len(cams), 1))(*cams) if cams else None
    buf = out if out is not None else np.empty(16, dtype=np.float32)
    st = vb.vk_stats()
    rc = getattr(ctx._L, fn)(ctx._h, arr, n, C.byref(p) if p is not None else None, buf.ctypes.data, C.byref(st))
    return rc, (ctx._L.vk_last_error(ctx._h) or b"").decode()


def test_batch_errors(vb, ctx):
    scene, cams = scene_and_cams(vb, "random_spheres_demo", 0, 3)
    fresh = vb.Context(0)
    p = vb.render_params(32, 18, 2, 10, seed=1)
    rc, msg = _raw(fresh, vb, cams, 3, p)
    assert rc == vb.VK_ERR_NO_SCENE, msg
    fresh.close()
    ctx.upload(scene)
    for fn in ("vk_render_frames", "vk_render_frames_rgb8"):
        assert _raw(ctx, vb, cams, 0, p, fn=fn)[0] == vb.VK_ERR_INVALID
        assert _raw(ctx, vb, [], 3, p, fn=fn)[0] == vb.VK_ERR_INVALID
        assert _raw(ctx, vb, cams, 3, None, fn=fn)[0] == vb.VK_ERR_INVALID
    bad = [vb.vk_camera.from_buffer_copy(c) for c in cams]
    bad[2].time0, bad[2].time1 = 1.0, 1.0
    rc, msg = _raw(ctx, vb, bad, 3, p)
    assert rc == vb.VK_ERR_INVALID and "frame 2" in msg, msg
    big = vb.render_params(8192, 8192, 1, 10, seed=1)  # 8192^2 * 3 * 11 > 2^31 - 1: refused before anything is allocated
    rc, msg = _raw(ctx, vb, cams * 4, 11, big)
    assert rc == vb.VK_ERR_INVALID and "too large" in msg, msg
    for v in (vb.VK_VARIANT_STAGED, vb.VK_VARIANT_WAVEFRONT):
        q = vb.render_params(32, 18, 2, 10, seed=1, variant=v)
        assert _raw(ctx, vb, cams, 3, q)[0] == vb.VK_ERR_UNSUPPORTED
        frame = np.empty(32 * 18 * 3, dtype=np.float32)
        assert _raw(ctx, vb, cams, 1, q, out=frame)[0] == 0  # one frame is vk_render: every variant
    # the context still renders after every refusal
    check_batch(vb, ctx, "random_spheres_demo", k=3)


def run_program(tmp_path, sub, *args):
    out = tmp_path / sub
    out.mkdir(exist_ok=True)
    r = subprocess.run([RENDER_BIN, "--out-dir", str(out)] + [str(a) for a in args], capture_output=True, text=True,
                       cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr
    return out, r.stderr


@pytest.mark.parametrize("extra", [[], ["--first-frame", 2]], ids=["from0", "first2"])
def test_program_batch_writes_the_same_files(tmp_path, extra):
    args = ["--scene", 3, "--width", 80, "--spp", 8, "--depth", 20, "--frames", 5] + extra
    a, ea = run_program(tmp_path, "one", *args, "--batch", 1)
    b, eb = run_program(tmp_path, "batch", *args, "--batch", 3)  # a batch of 3, then a short batch of 2
    names = sorted(os.listdir(a))
    assert len(names) == 5 and names == sorted(os.listdir(b))
    assert eb.count("Wrote frame") == 5
    for n in names:
        assert (a / n).read_bytes() == (b / n).read_bytes(), n
    assert (parse_ppm(str(a / names[0])) != parse_ppm(str(a / names[1]))).mean() > 0.05


@pytest.mark.parametrize("pin", [["--strict"], ["--variant", "stepq"]], ids=["strict", "variant"])
def test_program_batch_at_config1_size_writes_the_same_files(tmp_path, pin):
    # 400x225x16: one frame runs the lane megakernel under AUTO, a batch of 4 the step queues.  With --strict every kernel
    # computes the reference's operation sequence, with --variant both run the same kernel: the same bytes either way.
    args = ["--scene", 3, "--width", 400, "--spp", 16, "--depth", 50, "--frames", 4] + pin
    a, _ = run_program(tmp_path, "one", *args, "--batch", 1)
    b, _ = run_program(tmp_path, "batch", *args, "--batch", 4)
    names = sorted(os.listdir(a))
    assert len(names) == 4 and names == sorted(os.listdir(b))
    for n in names:
        assert (a / n).read_bytes() == (b / n).read_bytes(), n


def test_multi_gpu_batch_equals_the_one_gpu_batch(vb, ctx):
    try:
        m = vb.MultiContext([0, 1])
    except vb.VecchioError:
        pytest.skip("one GPU")
    for name, param in (("cornell_smoke", 0), ("random_spheres_demo", 0)):
        scene, cams = scene_and_cams(vb, name, param, 3)
        ctx.upload(scene)
        m.upload(scene)
        p = vb.render_params(96, scene.height_for(96), 33, 50, seed=4)
        a, sa = ctx.render_frames_rgb8(cams, p)
        b, sb = m.render_frames_rgb8(cams, p)
        assert np.array_equal(a, b) and (sa.paths, sa.rays) == (sb.paths, sb.rays)
    m.close()
