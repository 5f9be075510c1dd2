"""Adaptive render sessions on the GPU (vk_adaptive_*): a fresh session refined once equals the one-shot adaptive calls bit
for bit; any sequence of tightening targets ends bit for bit in the state of a fresh session refined once to the last one;
refusals, other calls on the context and a resume through export / import or a checkpoint change nothing they should not."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

_SCENES = {}


def scene_and_cams(vb, name, param=0, k=1):
    key = (name, param)
    if key not in _SCENES:
        s = vb.Scene(name, seed=1, param=param)
        base = s.next_camera()
        cams = [base]
        for f in range(1, 3):
            eye = [base.origin[i] + 0.3 * f * base.u[i] for i in range(3)]
            cams.append(vb.camera_new(eye, [eye[i] - base.w[i] for i in range(3)], list(base.v), 40.0, 1.0, 0.0, 10.0,
                                      base.time0, base.time1))
        _SCENES[key] = (s, cams)
    s, cams = _SCENES[key]
    return s, (cams[0] if k == 1 else cams[:k])


def params_like(p, **kw):
    q = type(p).from_buffer_copy(p)
    for k, v in kw.items():
        setattr(q, k, v)
    return q


def error_quantile(vb, ctx, cam, p, n, q=0.5):
    """A max_error that stops about a fraction q of the pixels at n samples (the header's rule on vk_render's sums)."""
    rgb, sq, _ = ctx.render(cam, params_like(p, spp=n, variant=0), want_sumsq=True)
    m = rgb.astype(np.float64)
    se = np.sqrt(np.maximum(sq.astype(np.float64) / n - m * m, 0.0) / (n - 1))
    e = (128.0 * (np.sqrt(np.maximum(m + se, 0.0)) - np.sqrt(np.maximum(m - se, 0.0)))).max(axis=-1)
    return max(float(np.quantile(e, q)), 0.01)


def state(sess):
    sums, sq, n, _ = sess.export()
    rgb, n1, e1 = sess.read()
    rgb8, n8, e8 = sess.read_rgb8()
    return [sums, sq, n, rgb, n1, e1, rgb8, n8, e8]


def assert_same(a, b, what=""):
    for i, (x, y) in enumerate(zip(a, b)):
        assert np.array_equal(x, y, equal_nan=x.dtype.kind == "f"), (what, i, int(np.sum(x != y)))


SCENES = [("cornell_box", 0), ("cornell_smoke", 0), ("random_spheres_demo", 0), ("bowser_demo", 0), ("final_scene", 0),
          ("api_surface_demo", 0), ("stress_spheres", 300)]


@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("strict", [False, True], ids=["render", "strict"])
@pytest.mark.parametrize("variant", ["AUTO", "WARPQ", "STEPQ", "MEGAKERNEL"])
@pytest.mark.parametrize("name,param", SCENES)
def test_fresh_session_refined_once_is_the_one_shot_call(vb, ctx, name, param, variant, strict, k):
    scene, cams = scene_and_cams(vb, name, param, k)
    ctx.upload(scene)
    p = vb.render_params(40, scene.height_for(40), 40, 30, seed=5, variant=getattr(vb, "VK_VARIANT_" + variant),
                         flags=vb.VK_FLAG_STRICT_MATH if strict else 0)
    E = error_quantile(vb, ctx, cams if k == 1 else cams[0], p, 8)
    sess = ctx.adaptive_session(cams, p, 8)
    st = sess.refine(E)
    rgb, n, _ = sess.read()
    rgb8, n8, _ = sess.read_rgb8()
    sess.close()
    if k == 1:
        w, wn, ws = ctx.render_adaptive(cams, p, 8, E)
        w8, wn8, _ = ctx.render_adaptive_rgb8(cams, p, 8, E)
    else:
        w, wn, ws = ctx.render_frames_adaptive(cams, p, 8, E)
        w8, wn8, _ = ctx.render_frames_adaptive_rgb8(cams, p, 8, E)
    assert np.array_equal(n, wn) and np.array_equal(rgb, w, equal_nan=True)
    assert np.array_equal(n8, wn8) and np.array_equal(rgb8, w8)
    assert st.paths == ws.paths == int(n.sum()) and st.variant == ws.variant
    assert len(np.unique(n)) >= 2


SEQUENCES = {
    "error": [dict(max_error=8.0), dict(max_error=4.0), dict(max_error=2.0), dict(max_error=1.0)],
    "cap": [dict(max_error=1.0, spp=64), dict(max_error=1.0, spp=128), dict(max_error=1.0, spp=256)],
    "floor": [dict(max_error=2.0, min_spp=0), dict(max_error=2.0, min_spp=128), dict(max_error=2.0, min_spp=256)],
    "mixed": [dict(max_error=6.0, spp=64), dict(max_error=3.0, spp=64, min_spp=32), dict(max_error=3.0, spp=192, min_spp=96),
              dict(max_error=0.0, spp=200, min_spp=96)],
    "repeat": [dict(max_error=2.0, spp=128, min_spp=64), dict(max_error=2.0, spp=128, min_spp=64)],
}
CASES = [("cornell_box", 0, 0), ("final_scene", 0, 0), ("cornell_smoke", 0, 0),
         ("random_spheres_cover", 0, "legacy_sky")]


def case_params(vb, scene, flags, width=48, spp=256, seed=7):
    f = vb.VK_FLAG_LEGACY_SCATTER | vb.VK_FLAG_SKY_BACKGROUND if flags == "legacy_sky" else 0
    return vb.render_params(width, scene.height_for(width), spp, 30, seed=seed, flags=f)


@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("seq", list(SEQUENCES))
@pytest.mark.parametrize("name,param,flags", CASES)
def test_tightening_sequence_equals_a_fresh_session_refined_once(vb, ctx, name, param, flags, seq, k):
    scene, cams = scene_and_cams(vb, name, param, k)
    ctx.upload(scene)
    p = case_params(vb, scene, flags)
    steps = SEQUENCES[seq]
    a = ctx.adaptive_session(cams, p, 32)
    before = None
    for i, t in enumerate(steps):
        sums0 = a.export()[2].astype(np.int64).sum()
        st = a.refine(**t)
        counts = a.export()[2]
        assert st.paths == int(counts.astype(np.int64).sum()) - sums0  # stats: samples added
        if seq == "repeat" and i == 1:
            assert st.paths == 0 and st.launches == 1  # (the level kernel only)
            assert_same(state(a), before, "repeat")
        before = state(a)
    b = ctx.adaptive_session(cams, p, 32)
    b.refine(**steps[-1])
    assert_same(state(a), state(b), seq)
    a.close()
    b.close()


def test_refusals_leave_the_state_byte_identical(vb, ctx):
    scene, cam = scene_and_cams(vb, "cornell_box")
    ctx.upload(scene)
    p = case_params(vb, scene, 0, spp=200)
    s = ctx.adaptive_session(cam, p, 32)
    s.refine(4.0, spp=100, min_spp=32)  # an off-grid cap: 100 is not a multiple of 32
    want = state(s)
    T = vb._abi.vk_adaptive_target
    bad = [T(100, 32, 8.0), T(100, 0, 4.0), T(96, 32, 4.0), T(128, 32, 4.0), T(201, 32, 4.0), T(0, 32, 4.0),
           T(100, 32, float("nan")), T(100, 32, -1.0)]
    for t in bad:  # straight to the library: the Python checks would refuse them first
        assert s._L.vk_adaptive_refine(s._h, t, None) == vb.VK_ERR_INVALID, (t.spp, t.min_spp, t.max_error)
        assert_same(state(s), want, (t.spp, t.min_spp, t.max_error))
    with pytest.raises(ValueError):
        s.refine(8.0, spp=100, min_spp=32)
    s2 = ctx.adaptive_session(cam, p, 32)
    s2.refine(0.0, spp=64)
    assert s2._L.vk_adaptive_refine(s2._h, T(64, 0, 1.0), None) == vb.VK_ERR_INVALID  # E > 0 after 0
    # a scene upload between refines
    ctx.upload(scene)
    with pytest.raises(vb.VecchioError, match="scene changed"):
        s.refine(2.0, spp=100, min_spp=32)
    assert_same(state(s), want, "scene")
    # an import with off-grid counts, or counts above the cap, or samples in a pixel with none counted
    sums, sq, n, r = s.export()
    for mutate in ("offgrid", "above", "zero"):
        n2, sums2 = n.copy(), sums.copy()
        at = np.unravel_index(np.argmax(sums.sum(axis=-1)), n.shape)  # a pixel with light in it
        n2[at] = {"offgrid": 33, "above": 128, "zero": 0}[mutate]
        with pytest.raises(vb.VecchioError, match="vk_adaptive_import"):
            s.import_(sums2, sq, n2, r)
        assert_same(state(s), want, mutate)
    s.close()
    s2.close()


def test_other_calls_on_the_context_do_not_touch_a_session(vb, ctx):
    scene, cams = scene_and_cams(vb, "random_spheres_demo", 0, 3)
    ctx.upload(scene)
    p = case_params(vb, scene, 0, spp=128)
    ref = ctx.adaptive_session(cams, p, 32)  # the same targets with nothing else run in between
    ref.refine(4.0)
    ref.refine(1.0)
    want = state(ref)
    ref.close()
    a = ctx.adaptive_session(cams, p, 32)
    b = ctx.adaptive_session(cams, p, 32)
    a.refine(4.0)
    b.refine(4.0)
    ctx.render(cams[0], params_like(p, spp=16, width=64, height=32))
    ctx.render_adaptive(cams[1], params_like(p, width=80, height=40), 16, 1.0)
    ctx.render_frames_adaptive(cams[::-1], p, 16, 1.0)  # (other cameras on the device, other counts in the staging)
    c = ctx.adaptive_session(cams[:2], params_like(p, width=96), 8)
    c.refine(2.0)
    a.refine(1.0)
    assert_same(state(a), want, "isolation: a")
    ctx.render_frames(cams[1:], params_like(p, spp=8))
    c.refine(1.0)
    b.refine(1.0)
    assert_same(state(b), want, "isolation: b")
    c.close()
    a.close()
    b.close()


def test_resume_in_a_new_context_equals_the_uninterrupted_sequence(vb, tmp_path):
    scene, cams = scene_and_cams(vb, "final_scene", 0, 3)
    steps = SEQUENCES["mixed"]
    ctx1 = vb.Context(0)
    ctx1.upload(scene)
    p = case_params(vb, scene, 0)
    full = ctx1.adaptive_session(cams, p, 32)
    for t in steps:
        full.refine(**t)
    want = state(full)
    half = ctx1.adaptive_session(cams, p, 32)
    half.refine(**steps[0])
    half.refine(**steps[1])
    saved = half.export()
    key = half.key("final_scene", 1)
    half.save(str(tmp_path / "ck.npz"), key)
    ctx1.close()  # (closes its sessions first)

    ctx2 = vb.Context(0)
    ctx2.upload(scene)
    r = ctx2.adaptive_session(cams, p, 32)
    r.import_(*saved)
    for t in steps[2:]:
        r.refine(**t)
    assert_same(state(r), want, "export / import")
    r2 = ctx2.adaptive_session(cams, p, 32)
    r2.load(str(tmp_path / "ck.npz"), key)
    assert r2.reached == saved[3]
    for t in steps[2:]:
        r2.refine(**t)
    assert_same(state(r2), want, "save / load")
    with pytest.raises(ValueError, match="another session"):
        r2.load(str(tmp_path / "ck.npz"), r2.key("final_scene", 2))
    other = ctx2.adaptive_session(cams, params_like(p, seed=p.seed + 1), 32)  # the checkpoint's own key, another session
    with pytest.raises(ValueError, match="not this session's identity"):
        other.load(str(tmp_path / "ck.npz"), key)
    assert other.export()[2].max() == 0
    other.close()
    # render_adaptive_resumable: an interrupted run (two targets) resumed with the whole list
    from vecchio_b200.adaptive_checkpoint import render_adaptive_resumable
    tl = [(t["max_error"], t.get("spp"), t.get("min_spp", 0)) for t in steps]
    ck = str(tmp_path / "run.npz")
    r3 = ctx2.adaptive_session(cams, p, 32)
    assert render_adaptive_resumable(r3, tl[:2], ck, key) == 2
    r4 = ctx2.adaptive_session(cams, p, 32)
    assert render_adaptive_resumable(r4, tl, ck, key) == 2
    assert_same(state(r4), want, "resumable")
    ctx2.close()


@pytest.mark.parametrize("name,param", [("final_scene", 0), ("cornell_box", 0)])
def test_floor(vb, ctx, name, param):
    scene, cam = scene_and_cams(vb, name, param)
    ctx.upload(scene)
    p = case_params(vb, scene, 0, spp=160)
    s = ctx.adaptive_session(cam, p, 32)
    s.refine(50.0, min_spp=70)
    _, _, n, _ = s.export()
    assert n.min() >= 96 and n.max() <= 160  # the first grid point >= 70
    s.close()
    s = ctx.adaptive_session(cam, p, 32)
    s.refine(50.0, spp=160, min_spp=160)  # a floor equal to the cap is the fixed render
    rgb, n, _ = s.read()
    want, _, _ = ctx.render(cam, params_like(p, spp=160, variant=s.variant))
    assert np.all(n == 160) and np.array_equal(rgb, want)
    s.close()


@pytest.mark.parametrize("name,param", [("cornell_smoke", 0), ("random_spheres_demo", 0)])
def test_error_map_and_stopped_pixels_obey_the_rule(vb, ctx, name, param):
    scene, cams = scene_and_cams(vb, name, param, 3)
    ctx.upload(scene)
    p = case_params(vb, scene, 0, spp=256)
    s = ctx.adaptive_session(cams, p, 32)
    E, floor = 2.0, 64
    s.refine(E, min_spp=floor)
    sums, sq, n, _ = s.export()
    _, n_read, err = s.read()
    assert np.array_equal(n, n_read)
    nd = n.astype(np.float64)[..., None]
    m = sums.astype(np.float64) * 2.0 ** -30 / nd
    q = sq.astype(np.float64) * 2.0 ** -32 / nd
    se = np.sqrt(np.maximum(q - m * m, 0.0) / (nd - 1))
    e = (128.0 * (np.sqrt(np.maximum(m + se, 0.0)) - np.sqrt(np.maximum(m - se, 0.0)))).max(axis=-1)
    close = np.abs(e - err) <= 0.01 * np.maximum(e, 1e-6)
    assert close.mean() > 0.999
    stopped = n < 256
    assert np.all(n[stopped] >= floor) and np.all(err[stopped] <= E * 1.0000001)
    _, n8, err8 = s.read_rgb8()
    assert np.array_equal(n8, n[:, ::-1]) and np.array_equal(err8, err[:, ::-1])
    s.close()
