"""Adaptive sampling split over shards of pixels, on the GPU: N shard sessions on one context add up, bit for bit, to the
unsharded session after one refine and after a tightening sequence; the summed state imported into a fresh session reads
exactly like the unsharded one; paths add up; pixels a shard does not own stay zero; an import that puts samples there is
refused and changes nothing; a shard checkpoint round-trips and never loads into a whole session.  With more than one
GPU, MultiContext's sessions and one-shot calls equal Context's on device 0, and an export of either resumes in the other."""
import numpy as np
import pytest

import shard_model as sm

pytestmark = pytest.mark.gpu

_SCENES = {}


def scene_and_cams(vb, name, k):
    if name not in _SCENES:
        s = vb.Scene(name, seed=1)
        cams = []
        while len(cams) < 16:
            c = s.next_camera()
            if c is None:
                break
            cams.append(c)
        base = cams[0]
        while len(cams) < 16:  # (scenes with one camera: views moved along u)
            eye = [base.origin[i] + 0.2 * len(cams) * base.u[i] for i in range(3)]
            cams.append(vb.camera_new(eye, [eye[i] - base.w[i] for i in range(3)], list(base.v), 40.0, 1.0, 0.0, 10.0,
                                      base.time0, base.time1))
        _SCENES[name] = (s, cams)
    s, cams = _SCENES[name]
    return s, (cams[0] if k == 1 else cams[:k])


def add(states):
    out = [np.zeros_like(a) for a in states[0][:3]]
    for st in states:
        for i in range(3):
            out[i] = out[i] + st[i]
    return out


def assert_same(a, b, what=""):
    for i, (x, y) in enumerate(zip(a, b)):
        assert x.dtype == y.dtype and np.array_equal(x, y, equal_nan=x.dtype.kind == "f"), (what, i, int(np.sum(x != y)))


def read_all(sess):
    return list(sess.read()) + list(sess.read_rgb8())


# (scene, K, width, cap spp, pass_spp, variant, strict, targets): a flat scene, media, and a BVH scene on the step queues
# (random spheres at bench config 1's 400x225, K = 16); both math builds; AUTO and explicit list-capable kernels
CASES = {
    "cornell-auto-render": ("cornell_box", 1, 64, 128, 16, "AUTO", False, [(128, 0, 6.0), (128, 0, 3.0), (128, 48, 3.0)]),
    "cornell-mega-strict": ("cornell_box", 3, 40, 96, 8, "MEGAKERNEL", True, [(48, 0, 4.0), (96, 0, 2.0)]),
    "smoke-warpq-render": ("cornell_smoke", 1, 72, 128, 16, "WARPQ", False, [(128, 0, 8.0), (128, 32, 4.0)]),
    "smoke-auto-strict": ("cornell_smoke", 3, 40, 64, 8, "AUTO", True, [(64, 0, 6.0), (64, 0, 3.0)]),
    "spheres16-auto-render": ("random_spheres_demo", 16, 400, 64, 16, "AUTO", False, [(64, 0, 4.0), (64, 0, 2.0)]),
    "spheres16-stepq-strict": ("random_spheres_demo", 16, 400, 48, 16, "STEPQ", True, [(32, 0, 4.0), (48, 0, 2.0)]),
}


def case(vb, ctx, name):
    scene_name, k, width, cap, M, variant, strict, targets = CASES[name]
    scene, cams = scene_and_cams(vb, scene_name, k)
    ctx.upload(scene)
    p = vb.render_params(width, scene.height_for(width), cap, 30, seed=11, variant=getattr(vb, "VK_VARIANT_" + variant),
                         flags=vb.VK_FLAG_STRICT_MATH if strict else 0)
    return scene, cams, p, M, targets


def refine(sess, t):
    return sess.refine(t[2], spp=t[0], min_spp=t[1])


@pytest.mark.parametrize("n_shards", [2, 3, 8])
@pytest.mark.parametrize("name", list(CASES))
def test_shard_exports_add_up_to_the_unsharded_session(vb, ctx, name, n_shards):
    scene, cams, p, M, targets = case(vb, ctx, name)
    whole = ctx.adaptive_session(cams, p, M)
    shards = [ctx.adaptive_session(cams, p, M, shard=(k, n_shards)) for k in range(n_shards)]
    assert all(s.variant == whole.variant for s in shards)  # (AUTO decides on the whole batch)
    shape = whole.export()[2].shape
    for step, t in enumerate(targets):
        sw = refine(whole, t)
        ss = [refine(s, t) for s in shards]
        want = whole.export()
        got = [s.export() for s in shards]
        for k, g in enumerate(got):
            mine = sm.owned(shape, k, n_shards)
            assert not g[0][~mine].any() and not g[1][~mine].any() and not g[2][~mine].any(), (step, k)
            assert g[3] == want[3]
        assert_same(add(got), want[:3], (name, n_shards, step))
        assert sum(s.paths for s in ss) == sw.paths and all(s.variant == sw.variant for s in ss)
        if step == 0:  # the first target is the one-shot call's
            assert len(np.unique(want[2])) >= 2
            fresh = ctx.adaptive_session(cams, p, M)
            fresh.import_(*add(got), want[3])
            got_read, want_read = read_all(fresh), read_all(whole)
            assert_same(got_read, want_read, "imported sum")
            fresh.close()
            one = ctx.render_adaptive_rgb8 if len(shape) == 2 else ctx.render_frames_adaptive_rgb8
            if t[1] == 0 and t[0] == p.spp:
                rgb8, cnt, _ = one(cams, p, M, t[2])
                assert np.array_equal(rgb8, want_read[3]) and np.array_equal(cnt, want_read[4])
    for s in shards:
        s.close()
    whole.close()


def test_a_shard_refuses_samples_on_pixels_it_does_not_own_and_round_trips_its_checkpoint(vb, ctx, tmp_path):
    scene, cams, p, M, targets = case(vb, ctx, "smoke-auto-strict")
    s = ctx.adaptive_session(cams, p, M, shard=(1, 3))
    refine(s, targets[0])
    before = s.export()
    reads = read_all(s)
    shape = before[2].shape
    mine = sm.owned(shape, 1, 3)
    other = np.flatnonzero(~mine.reshape(-1))[5]
    for what in range(3):
        bad = [a.copy() for a in before[:3]]
        if what == 2:
            bad[2].reshape(-1)[other] = M
        else:
            bad[what].reshape(-1, 3)[other, 0] = 1
        with pytest.raises(vb.VecchioError, match="not this shard's"):
            s.import_(*bad, before[3])
        assert_same(s.export()[:3], before[:3], ("refused import", what))
    assert_same(read_all(s), reads, "untouched")
    # what reads for a pixel the shard does not own: count 0, mean NaN, rgb8 0, error +inf
    rgb, n, e, rgb8, n8, e8 = reads
    assert (n[~mine] == 0).all() and np.isnan(rgb[~mine]).all() and np.isinf(e[~mine]).all()
    assert (n8 == 0).sum() == (~mine).sum() and (rgb8[n8 == 0] == 0).all()
    path = str(tmp_path / "shard.npz")
    key = s.key(scene.name, 1)
    assert key["shard"] == [1, 3]
    s.save(path, key)
    again = ctx.adaptive_session(cams, p, M, shard=(1, 3))
    again.load(path, key)
    assert_same(again.export()[:3], before[:3], "checkpoint")
    assert again.reached == s.reached
    refine(again, targets[1])
    refine(s, targets[1])
    assert_same(again.export()[:3], s.export()[:3], "resumed")
    whole = ctx.adaptive_session(cams, p, M)
    with pytest.raises(ValueError, match="not this session's identity"):
        whole.load(path, key)
    with pytest.raises(ValueError, match="another session"):
        whole.load(path, whole.key(scene.name, 1))
    for x in (s, again, whole):
        x.close()


def test_a_shard_without_pixels_renders_nothing_and_reaches_its_target(vb, ctx):
    scene, cams = scene_and_cams(vb, "cornell_box", 1)
    ctx.upload(scene)
    p = vb.render_params(8, 6, 64, 30, seed=3)  # 48 pixels: two runs
    s = ctx.adaptive_session(cams, p, 16, shard=(2, 3))
    st = s.refine(4.0)
    assert st.paths == 0 and st.launches == 0 and s.reached == s.target(4.0)
    st = s.refine(2.0)
    assert st.paths == 0 and st.launches == 0
    sums, sq, n, reached = s.export()
    assert not sums.any() and not sq.any() and not n.any() and reached == s.target(2.0)
    s.close()
    for bad in ((3, 3), (0, 0)):
        with pytest.raises(ValueError):
            ctx.adaptive_session(cams, p, 16, shard=bad)


# ---- several GPUs ----

def multi_or_skip(vb):
    try:
        return vb.MultiContext(list(range(max(2, min(8, _device_count())))))
    except vb.VecchioError:
        pytest.skip("one GPU")


def _device_count():
    from conftest import cuda_device_count
    return cuda_device_count()


@pytest.mark.parametrize("name", ["cornell-auto-render", "smoke-auto-strict", "spheres16-auto-render"])
def test_multi_context_adaptive_equals_the_one_gpu_session(vb, ctx, name):
    m = multi_or_skip(vb)
    scene, cams, p, M, targets = case(vb, ctx, name)
    m.upload(scene)
    one = ctx.adaptive_session(cams, p, M)
    many = m.adaptive_session(cams, p, M)
    assert many.variant == one.variant
    for t in targets:
        s1, s2 = refine(one, t), refine(many, t)
        assert s1.paths == s2.paths and s1.variant == s2.variant
        assert_same(many.export()[:3], one.export()[:3], (name, t))
        assert_same(read_all(many), read_all(one), (name, t))
    # an export of either resumes in the other, in both directions
    a = m.adaptive_session(cams, p, M)
    a.import_(*one.export())
    b = ctx.adaptive_session(cams, p, M)
    b.import_(*many.export())
    assert a.key(scene.name, 1) == b.key(scene.name, 1)
    last = (p.spp, targets[-1][1], targets[-1][2] / 2)
    for x in (a, b, one):
        refine(x, last)
    assert_same(a.export()[:3], one.export()[:3], "one -> many")
    assert_same(b.export()[:3], one.export()[:3], "many -> one")
    t0 = targets[0]
    if t0[0] == p.spp and t0[1] == 0:
        if isinstance(cams, list):
            w8, wn, ws = ctx.render_frames_adaptive_rgb8(cams, p, M, t0[2])
            g8, gn, gs = m.render_frames_adaptive_rgb8(cams, p, M, t0[2])
        else:
            w8, wn, ws = ctx.render_adaptive_rgb8(cams, p, M, t0[2])
            g8, gn, gs = m.render_adaptive_rgb8(cams, p, M, t0[2])
        assert np.array_equal(w8, g8) and np.array_equal(wn, gn) and ws.paths == gs.paths and ws.variant == gs.variant
    for x in (one, many, a, b):
        x.close()
    m.close()
