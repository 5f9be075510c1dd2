"""The end of every render call into host buffers (the readout in vk_api.cu): one conversion launch on top of the render's
own launches, a batch of one frame that is the one-frame call, rgb8 batches that are frame_to_rgb8 of the float batch, and
MultiContext's fixed renders counted and converted like one GPU's."""
import numpy as np
import pytest

from conftest import cuda_device_count

pytestmark = pytest.mark.gpu

SCENES = ["cornell_box", "random_spheres_demo"]


def scene_and_cam(vb, name):
    scene = vb.Scene(name, seed=1)
    return scene, scene.next_camera()


def with_seed(p, seed):
    q = type(p).from_buffer_copy(p)
    q.seed = seed
    return q


def device_launches(ctx, cam, p):
    torch = pytest.importorskip("torch")
    d_sum = torch.empty(p.width * p.height * 3, dtype=torch.float32, device=f"cuda:{ctx.device}")
    ctx.flush_stats()  # (launches an earlier test left uncounted would land in the first count)
    return ctx.render_device(cam, p, d_sum.data_ptr()).launches


@pytest.mark.parametrize("variant", ["AUTO", "MEGAKERNEL"])
@pytest.mark.parametrize("name", SCENES)
def test_host_renders_report_the_device_render_plus_one_conversion(vb, ctx, name, variant):
    scene, cam = scene_and_cam(vb, name)
    ctx.upload(scene)
    p = vb.render_params(61, 37, 12, 20, seed=3, variant=getattr(vb, "VK_VARIANT_" + variant))
    want = device_launches(ctx, cam, p) + 1
    assert ctx.render(cam, p)[2].launches == want
    assert ctx.render(cam, p, want_sumsq=True)[2].launches == want
    assert ctx.render_rgb8(cam, p)[1].launches == want
    for k in (1, 3):  # a batch is one launch over all its frames
        assert ctx.render_frames([cam] * k, p)[1].launches == want, k
        assert ctx.render_frames_rgb8([cam] * k, p)[1].launches == want, k


@pytest.mark.parametrize("variant", ["AUTO", "STAGED", "WAVEFRONT", "MEGAKERNEL"])
@pytest.mark.parametrize("name", SCENES)
def test_a_batch_of_one_frame_is_the_one_frame_call(vb, ctx, name, variant):
    scene, cam = scene_and_cam(vb, name)
    ctx.upload(scene)
    p = vb.render_params(61, 37, 10, 20, seed=5, variant=getattr(vb, "VK_VARIANT_" + variant))
    a, _, sa = ctx.render(cam, p)
    b, sb = ctx.render_frames([cam], p)
    assert b.shape == (1,) + a.shape and np.array_equal(a, b[0])
    assert (sa.paths, sa.rays, sa.launches, sa.variant) == (sb.paths, sb.rays, sb.launches, sb.variant)
    a8, sa8 = ctx.render_rgb8(cam, p)
    b8, sb8 = ctx.render_frames_rgb8([cam], p)
    assert np.array_equal(a8, b8[0]) and np.array_equal(a8, vb.frame_to_rgb8(a))
    assert (sa8.paths, sa8.rays, sa8.launches) == (sb8.paths, sb8.rays, sb8.launches)


@pytest.mark.parametrize("name", SCENES)
def test_rgb8_batch_is_frame_to_rgb8_of_the_float_batch(vb, ctx, name):
    scene, cam = scene_and_cam(vb, name)
    ctx.upload(scene)
    p = vb.render_params(61, 37, 8, 20, seed=7)  # ragged: no dimension a multiple of 4, a plane not a multiple of 4 bytes
    frames, _ = ctx.render_frames([cam] * 3, p)
    rgb8, _ = ctx.render_frames_rgb8([cam] * 3, p)
    assert rgb8.shape == (3, 37, 61, 3)
    for f in range(3):
        assert np.array_equal(rgb8[f], vb.frame_to_rgb8(frames[f])), f
        assert np.array_equal(frames[f], ctx.render(cam, with_seed(p, p.seed + f))[0]), f


# A fixed render on a MultiContext launches the lane megakernel once per device (each renders its slice of the samples),
# then k_reduce_peers and the conversion on device 0.
MULTI_LAUNCHES_PER_DEVICE = 1
MULTI_LAUNCHES_ON_DEVICE_0 = 2


@pytest.mark.parametrize("name", SCENES)
def test_multi_context_readout_counts_and_converts_like_one_gpu(vb, ctx, name):
    n = min(8, cuda_device_count())
    if n < 2:
        pytest.skip("one GPU")
    m = vb.MultiContext(list(range(n)))
    want_launches = n * MULTI_LAUNCHES_PER_DEVICE + MULTI_LAUNCHES_ON_DEVICE_0
    scene, cam = scene_and_cam(vb, name)
    ctx.upload(scene)
    m.upload(scene)
    p = vb.render_params(61, 37, 16, 20, seed=9, variant=vb.VK_VARIANT_MEGAKERNEL)
    a, _, sa = ctx.render(cam, p)
    b, _, sb = m.render(cam, p)
    assert np.array_equal(a, b) and (sa.paths, sa.rays) == (sb.paths, sb.rays) and sb.launches == want_launches
    b, _, sb = m.render(cam, p, want_sumsq=True)
    assert np.array_equal(a, b) and (sa.paths, sa.rays) == (sb.paths, sb.rays) and sb.launches == want_launches
    a8, sa8 = ctx.render_rgb8(cam, p)
    b8, sb8 = m.render_rgb8(cam, p)
    assert np.array_equal(a8, b8) and (sa8.paths, sa8.rays) == (sb8.paths, sb8.rays) and sb8.launches == want_launches
    for k in (1, 3):
        a8, sa8 = ctx.render_frames_rgb8([cam] * k, p)
        b8, sb8 = m.render_frames_rgb8([cam] * k, p)
        assert np.array_equal(a8, b8) and (sa8.paths, sa8.rays) == (sb8.paths, sb8.rays), k
        assert sb8.launches == want_launches, k
    m.close()
