"""The render inputs no shipped scene uses, through every kernel and work domain: a thin-lens camera, a shutter other than
[0, 1], a non-black constant background, the sky under HEAD's integrator, depths 2 to 5, seeds of 2^32 and more, and
depth 0 (refused).

Each input is checked three ways: the render build against the oracle (the bars of test_image_parity_3_sigma), every
variant's strict-build frame against the lane megakernel's bit for bit (the rule of test_variants_equal_megakernel), and
in the other work domains (a batch of frames, an adaptive render's pixel lists).  The generation stage -- jitter, the
(width - 1) divisor, the lens law, the u/v offsets -- is also checked against a closed form that does not use the oracle:
at depth 1 on cornell_box a sample is 15 exactly when the camera ray's first hit is the light, so a pixel's count of
such samples is binomial with the share p of its footprint (averaged over the lens) that sees the light."""
import subprocess

import numpy as np
import pytest
from scipy import stats as sst

from conftest import ROOT, cuda_device_count, get_scene
from test_frames_and_checkpoints import RENDER_BIN
from test_gpu_parity import zscores
from test_zz_adaptive_gpu import median_error_target, on_pass_grid, params_like
from test_zz_batch_frames_gpu import singles

gpu = pytest.mark.gpu
BACKGROUND = (0.2, 0.3, 0.5)


def view(vb, cam, aperture=0.0, focus=None, time0=None, time1=None):
    """cam's view (eye, direction, up, field of view, aspect) rebuilt by Camera::new with another lens and shutter."""
    f = lambda a: np.array(a[:], dtype=np.float64)  # noqa: E731
    o, llc, h, v, w = f(cam.origin), f(cam.lower_left_corner), f(cam.horizontal), f(cam.vertical), f(cam.w)
    dist = -np.dot(llc + h / 2 + v / 2 - o, w)  # the focus distance cam was built with
    vfov = np.degrees(2 * np.arctan(np.linalg.norm(v) / 2 / dist))
    return vb.camera_new(o, o - w, f(cam.v), vfov, np.linalg.norm(h) / np.linalg.norm(v), aperture,
                         dist if focus is None else focus, cam.time0 if time0 is None else time0,
                         cam.time1 if time1 is None else time1)


# ---------------------------------------------------------------------------------------------------------------------
# Against the oracle, across the variants, and the Cornell static-shape kernel
# ---------------------------------------------------------------------------------------------------------------------
FLAT = {"cornell_box", "cornell_smoke"}
# (id, scene, camera(vb, cam), width, spp, depth, flags, background); the oracle renders at most ~2 M paths
LENS_CORNELL = lambda vb, c: view(vb, c, aperture=60.0, focus=1100.0)  # noqa: E731
CASES = [("lens_cornell_box", "cornell_box", LENS_CORNELL, 64, 512, 50, 0, None),
         ("lens_random_spheres", "random_spheres_demo", lambda vb, c: view(vb, c, aperture=0.5, focus=10.0), 96, 256, 50, 0, None),
         ("lens_final_scene", "final_scene", lambda vb, c: view(vb, c, aperture=20.0, focus=500.0), 48, 512, 50, 0, None),
         ("shutter_final_scene", "final_scene", lambda vb, c: view(vb, c, time0=0.25, time1=0.5), 48, 512, 50, 0, None),
         ("background_cornell_box", "cornell_box", None, 64, 512, 50, 0, BACKGROUND),
         ("background_random_spheres", "random_spheres_demo", None, 96, 256, 50, 0, BACKGROUND),
         ("sky_cornell_box", "cornell_box", None, 64, 512, 50, "sky", None),
         ("sky_random_spheres", "random_spheres_demo", None, 96, 256, 50, "sky", None)]
CASES += [(f"depth{d}_{n}", n, None, W, spp, d, 0, None)
          for d in (2, 3, 5) for n, W, spp in (("cornell_box", 64, 512), ("cornell_smoke", 64, 512), ("random_spheres_demo", 96, 256))]


def case_inputs(vb, name, camf, flags, bg):
    scene, cam = get_scene(vb, name)
    cam = camf(vb, cam) if camf else cam
    f = vb.VK_FLAG_SKY_BACKGROUND if flags == "sky" else flags
    return scene, cam, f, (bg or (0.0, 0.0, 0.0))


def check_oracle_bars(vb, po, ctx, label, scene, cam, W, spp, depth, flags, bg):
    """test_image_parity_3_sigma's bars: per pixel-channel z, 8x8 tiles, image mean, segments per path."""
    H = scene.height_for(W)
    o = po.OracleScene(scene)
    ro, qo, so = o.render(cam, vb.render_params(W, H, spp, depth, seed=21, flags=flags, background=bg), want_sumsq=True)
    rg, qg, sg = ctx.render(cam, vb.render_params(W, H, spp, depth, seed=22, flags=flags, background=bg), want_sumsq=True)
    assert np.isfinite(rg).all() and sg.paths == W * H * spp
    seg_g, seg_o = sg.rays / sg.paths, so.rays_live / so.paths
    z, nz, diff, se = zscores(rg, qg, spp, ro, qo, spp)
    frac = (np.abs(z[nz]) <= 3.0).mean()
    th, tw = H // 8, W // 8
    dt = diff[: th * 8, : tw * 8].reshape(th, 8, tw, 8, 3).sum(axis=(1, 3))
    st = np.sqrt((se[: th * 8, : tw * 8] ** 2).reshape(th, 8, tw, 8, 3).sum(axis=(1, 3)))
    zt = dt[st > 0] / st[st > 0]
    ztile = np.where(st > 0, np.abs(dt) / np.where(st > 0, st, 1.0), 0.0).max(axis=2)
    print(f"{label} (variant {sg.variant}): {frac:.4f} of {int(nz.sum())} pixel-channels within 3 sigma, mean z {z[nz].mean():+.3f}, "
          f"tiles within 3 sigma {(np.abs(zt) <= 3).mean():.4f}, image mean ratio {rg.mean() / ro.mean():.4f}, "
          f"segments per path {seg_g:.4f} (oracle, live {seg_o:.4f})")
    assert abs(seg_g - seg_o) <= 0.02 * seg_o, (label, seg_g, seg_o)
    assert frac >= 0.985, (label, frac)
    assert abs(z[nz].mean()) <= 0.1, (label, z[nz].mean())
    assert np.isfinite(z[~nz]).all(), "a pixel is constant in both renders but differs"
    assert (np.abs(zt) <= 3).mean() >= 0.98 and (ztile > 6.0).sum() <= 1, (label, (np.abs(zt) <= 3).mean(), np.abs(zt).max())
    assert abs(rg.mean() - ro.mean()) <= 0.01 * ro.mean(), (label, rg.mean(), ro.mean())


def strict_frame(vb, ctx, cam, W, H, spp, depth, flags, bg, variant, seed=31):
    p = vb.render_params(W, H, spp, depth, seed=seed, variant=variant, flags=flags | vb.VK_FLAG_STRICT_MATH, background=bg)
    return ctx.render(cam, p)


def check_variants_equal_megakernel(vb, ctx, monkeypatch, label, name, scene, cam, depth, flags, bg):
    """Strict build: every variant that runs the scene renders the lane megakernel's frame with its ray and dropped-sample
    counts.  On final_scene also the dynamic megakernel and the lane megakernel over the hybrid program."""
    W, spp = 48, 16
    H = scene.height_for(W)
    a, _, sa = strict_frame(vb, ctx, cam, W, H, spp, depth, flags, bg, vb.VK_VARIANT_MEGAKERNEL)
    assert sa.variant == vb.VK_VARIANT_MEGAKERNEL
    variants = ([vb.VK_VARIANT_WAVEFRONT, vb.VK_VARIANT_STAGED, vb.VK_VARIANT_WARPQ] if name in FLAT
                else [vb.VK_VARIANT_WAVEFRONT, vb.VK_VARIANT_WARPQ, vb.VK_VARIANT_STEPQ])
    for v in variants:
        b, _, sb = strict_frame(vb, ctx, cam, W, H, spp, depth, flags, bg, v)
        assert sb.variant == v and sb.paths == sa.paths, (label, v, sb.variant)
        assert np.array_equal(a, b), (label, v, np.abs(a - b).max())
        assert (sa.rays, sa.dropped_samples) == (sb.rays, sb.dropped_samples), (label, v)
    if name == "final_scene":
        monkeypatch.setenv("VECCHIO_MEGA", "dynamic")
        b, _, sb = strict_frame(vb, ctx, cam, W, H, spp, depth, flags, bg, vb.VK_VARIANT_MEGAKERNEL)
        monkeypatch.delenv("VECCHIO_MEGA")
        assert np.array_equal(a, b) and (sa.rays, sa.dropped_samples) == (sb.rays, sb.dropped_samples), (label, "dynamic")
        monkeypatch.setenv("VECCHIO_HYBRID_ALL", "1")
        b, _, sb = strict_frame(vb, ctx, cam, W, H, spp, depth, flags, bg, vb.VK_VARIANT_MEGAKERNEL)
        monkeypatch.delenv("VECCHIO_HYBRID_ALL")
        # (test_hybrid_program_renders_the_same_image's rule: exact ties between a subtree and the flat top may resolve
        # differently)
        assert np.array_equal(a, b) or np.isclose(a, b, rtol=1e-5, atol=1e-6).mean() > 0.999, (label, "hybrid")


def check_static_shape_kernel(vb, ctx, monkeypatch, label, scene, cam, depth, flags, bg):
    """Render build on cornell_box: the kernel compiled for the flat program's shape renders the generic kernel's bytes."""
    assert vb.scene_check(scene.desc_ptr)["flat_shape"] != 0
    p = vb.render_params(96, 96, 24, depth, seed=5, variant=vb.VK_VARIANT_WARPQ, flags=flags, background=bg)
    a, qa, sa = ctx.render(cam, p, want_sumsq=True)
    monkeypatch.setenv("VECCHIO_NO_STATIC_FLAT", "1")
    b, qb, sb = ctx.render(cam, p, want_sumsq=True)
    monkeypatch.delenv("VECCHIO_NO_STATIC_FLAT")
    assert a.tobytes() == b.tobytes() and np.array_equal(qa, qb), label
    assert (sa.paths, sa.rays, sa.dropped_samples) == (sb.paths, sb.rays, sb.dropped_samples), label


@gpu
@pytest.mark.parametrize("label,name,camf,W,spp,depth,flags,bg", CASES, ids=[c[0] for c in CASES])
def test_render_input(vb, po, ctx, monkeypatch, label, name, camf, W, spp, depth, flags, bg):
    scene, cam, f, bg = case_inputs(vb, name, camf, flags, bg)
    ctx.upload(scene)
    check_oracle_bars(vb, po, ctx, label, scene, cam, W, spp, depth, f, bg)
    check_variants_equal_megakernel(vb, ctx, monkeypatch, label, name, scene, cam, depth, f, bg)
    if name == "cornell_box":
        check_static_shape_kernel(vb, ctx, monkeypatch, label, scene, cam, depth, f, bg)


# ---------------------------------------------------------------------------------------------------------------------
# Work domains (strict build): a batch of frames, an adaptive render's pixel lists
# ---------------------------------------------------------------------------------------------------------------------
def batch_cams(vb, name):
    """Three cameras of one view, each with another lens and shutter."""
    _, cam = get_scene(vb, name)
    big = 60.0 if name in FLAT else 20.0
    return [view(vb, cam, aperture=big, time0=0.0, time1=1.0), view(vb, cam, aperture=big / 4, time0=0.25, time1=0.5),
            view(vb, cam, aperture=0.0, time0=0.5, time1=0.75)]


@gpu
@pytest.mark.parametrize("bg", [(0.0, 0.0, 0.0), BACKGROUND], ids=["black", "background"])
@pytest.mark.parametrize("variant", ["AUTO", "WARPQ", "STEPQ", "MEGAKERNEL"])
@pytest.mark.parametrize("name", ["cornell_box", "final_scene"])
def test_batch_of_lens_and_shutter_cameras_equals_single_frames(vb, ctx, name, variant, bg):
    scene, _ = get_scene(vb, name)
    cams = batch_cams(vb, name)
    ctx.upload(scene)
    W = 64
    p = vb.render_params(W, scene.height_for(W), 8, 30, seed=11, variant=getattr(vb, "VK_VARIANT_" + variant),
                         flags=vb.VK_FLAG_STRICT_MATH, background=bg)
    got, st = ctx.render_frames(cams, p)
    want, sts = singles(ctx, cams, p)
    assert np.array_equal(got, want), (name, variant, bg)
    assert st.paths == sum(s.paths for s in sts) and st.rays == sum(s.rays for s in sts)
    assert st.dropped_samples == sum(s.dropped_samples for s in sts)
    assert not np.array_equal(got[0], got[1]) and not np.array_equal(got[1], got[2])


@gpu
@pytest.mark.parametrize("variant", ["AUTO", "WARPQ", "STEPQ", "MEGAKERNEL"])
@pytest.mark.parametrize("name,aperture,focus", [("cornell_box", 60.0, 1100.0), ("random_spheres_demo", 0.5, 10.0)])
def test_adaptive_lens_pixels_equal_fixed_renders_at_their_count(vb, ctx, name, aperture, focus, variant):
    scene, cam = get_scene(vb, name)
    cam = view(vb, cam, aperture=aperture, focus=focus)
    ctx.upload(scene)
    W, spp, pass_spp = 64, 40, 8
    p = vb.render_params(W, scene.height_for(W), spp, 30, seed=11, variant=getattr(vb, "VK_VARIANT_" + variant),
                         flags=vb.VK_FLAG_STRICT_MATH)
    rgb, n, st = ctx.render_adaptive(cam, p, pass_spp, median_error_target(vb, ctx, cam, p, pass_spp))
    assert on_pass_grid(n, pass_spp, spp) and len(np.unique(n)) >= 2, (name, np.unique(n))
    assert st.paths == int(n.sum(dtype=np.uint64))
    q = params_like(vb, p, variant=st.variant)
    for v in np.unique(n):
        want, _, sw = ctx.render(cam, params_like(vb, q, spp=int(v)))
        assert sw.variant == st.variant
        assert np.array_equal(rgb[n == v], want[n == v]), (name, int(v))


# ---------------------------------------------------------------------------------------------------------------------
# Seeds of 2^32 and more
# ---------------------------------------------------------------------------------------------------------------------
SEED_VARIANTS = {"cornell_box": ["AUTO", "MEGAKERNEL", "WAVEFRONT", "STAGED", "WARPQ"],
                 "random_spheres_demo": ["AUTO", "MEGAKERNEL", "WAVEFRONT", "STAGED", "WARPQ", "STEPQ"]}


@gpu
@pytest.mark.parametrize("strict", [False, True], ids=["render", "strict"])
@pytest.mark.parametrize("name", list(SEED_VARIANTS))
def test_seed_high_word_changes_the_frame(vb, ctx, name, strict):
    """Philox's key is the whole 64-bit seed: s and s + 2^32 are different frames in every variant."""
    scene, cam = get_scene(vb, name)
    ctx.upload(scene)
    for v in SEED_VARIANTS[name]:
        p = lambda seed: vb.render_params(48, scene.height_for(48), 4, 20, seed=seed, variant=getattr(vb, "VK_VARIANT_" + v),  # noqa: E731
                                          flags=vb.VK_FLAG_STRICT_MATH if strict else 0)
        a, _, _ = ctx.render(cam, p(7))
        b, _, _ = ctx.render(cam, p(7 + (1 << 32)))
        c, _, _ = ctx.render(cam, p(7 + (1 << 32)))
        assert np.array_equal(b, c) and (a != b).mean() > 0.3, (name, v, (a != b).mean())


@gpu
@pytest.mark.parametrize("variant", ["AUTO", "WARPQ", "STEPQ", "MEGAKERNEL"])
@pytest.mark.parametrize("name", ["cornell_box", "random_spheres_demo"])
def test_batch_key_carries_into_the_high_word(vb, ctx, name, variant):
    """Frame f of a batch uses key seed + f as a 64-bit sum: from 2^32 - 1, frame 1 is the single render at 2^32."""
    scene, cam = get_scene(vb, name)
    ctx.upload(scene)
    W = 48
    p = vb.render_params(W, scene.height_for(W), 8, 20, seed=(1 << 32) - 1, variant=getattr(vb, "VK_VARIANT_" + variant),
                         flags=vb.VK_FLAG_STRICT_MATH)
    got, _ = ctx.render_frames([cam, cam], p)
    lo, _, _ = ctx.render(cam, params_like(vb, p, seed=(1 << 32) - 1))
    hi, _, _ = ctx.render(cam, params_like(vb, p, seed=1 << 32))
    wrap, _, _ = ctx.render(cam, params_like(vb, p, seed=0))
    assert np.array_equal(got[0], lo) and np.array_equal(got[1], hi), (name, variant)
    assert not np.array_equal(got[1], wrap)


# ---------------------------------------------------------------------------------------------------------------------
# Depth 0: refused by every render call (ray_color starts at depth 1; 0 would be a black frame with no rays)
# ---------------------------------------------------------------------------------------------------------------------
def assert_refuses_depth0(vb, call):
    with pytest.raises(vb.VecchioError) as e:
        call()
    assert e.value.code == vb.VK_ERR_INVALID and "max_depth" in str(e.value) and "main.rs:126" in str(e.value), str(e.value)


@gpu
def test_depth_zero_is_refused_everywhere(vb, ctx, tmp_path):
    scene, cam = get_scene(vb, "cornell_box")
    ctx.upload(scene)
    p = vb.render_params(32, 32, 8, 0, seed=1)
    calls = {"render": lambda c: c.render(cam, p), "render_rgb8": lambda c: c.render_rgb8(cam, p),
             "render_frames": lambda c: c.render_frames([cam, cam], p),
             "render_adaptive": lambda c: c.render_adaptive(cam, p, 4, 1.0),
             "render_frames_adaptive": lambda c: c.render_frames_adaptive([cam, cam], p, 4, 1.0),
             "adaptive_session": lambda c: c.adaptive_session(cam, p, 4)}
    for who, call in calls.items():
        assert_refuses_depth0(vb, lambda: call(ctx))
        print(f"depth 0 refused: Context.{who}")
    ctx.render(cam, params_like(vb, p, max_depth=1))  # depth 1 renders
    if cuda_device_count() >= 2:
        m = vb.MultiContext([0, 1])
        try:
            m.upload(scene)
            for who, call in {"render": lambda: m.render(cam, p), "render_rgb8": lambda: m.render_rgb8(cam, p),
                              "render_frames_rgb8": lambda: m.render_frames_rgb8([cam, cam], p),
                              "render_adaptive_rgb8": lambda: m.render_adaptive_rgb8(cam, p, 4, 1.0),
                              "adaptive_session": lambda: m.adaptive_session(cam, p, 4)}.items():
                assert_refuses_depth0(vb, call)
                print(f"depth 0 refused: MultiContext.{who}")
        finally:
            m.close()
    out = tmp_path / "frames"
    out.mkdir()
    r = subprocess.run([RENDER_BIN, "--out-dir", str(out), "--width", "32", "--spp", "4", "--depth", "0"], capture_output=True,
                       text=True, cwd=ROOT, timeout=600)
    assert r.returncode != 0 and "max_depth" in r.stderr and "main.rs:126" in r.stderr, (r.returncode, r.stderr)
    assert not list(out.iterdir())
    print(f"depth 0 refused: vecchio_gpu_render ({r.stderr.strip()})")


# ---------------------------------------------------------------------------------------------------------------------
# The generation stage against a closed form (no oracle): depth 1 on cornell_box
# ---------------------------------------------------------------------------------------------------------------------
# The light (src/scene.rs, cornell_box): XZRect x 213..343, z 227..332 at y = 554, under the ceiling at 555; the tall box
# ends at y = 330 and the front of the room is open, so nothing blocks a camera ray on its way up to the light.
LIGHT = np.array([[213.0, 554.0, 227.0], [343.0, 554.0, 227.0], [343.0, 554.0, 332.0], [213.0, 554.0, 332.0]])
CF_W, CF_H, CF_SPP = 97, 61, 4096


def cf_camera(vb, aperture):
    """Looking up at the light from the room's usual eye; at aperture 30 the light's edges blur over ~3 pixels."""
    return vb.camera_new([278, 278, -800], [278, 554, 280], [0, 1, 0], 10.0, CF_W / CF_H, aperture, 700.0, 0.0, 1.0)


def light_quad(cam, W, H, lens_xy):
    """The light's preimage in pixel coordinates (s (W-1), t (H-1)) for a ray leaving the lens at lens_xy: the rect's
    corners projected from the ray's origin onto the plane llc + s horizontal + t vertical."""
    f = lambda a: np.array(a[:], dtype=np.float64)  # noqa: E731
    o = f(cam.origin) + f(cam.u) * lens_xy[0] + f(cam.v) * lens_xy[1]
    h, v, llc = f(cam.horizontal), f(cam.vertical), f(cam.lower_left_corner)
    q = []
    for c in LIGHT:
        s, t, _ = np.linalg.solve(np.stack([h, v, -(c - o)], axis=1), o - llc)
        q.append((s * (W - 1), t * (H - 1)))
    return np.array(q)


def box_quad_area(quad, x0, x1, y0, y1):
    """Area of [x0, x1] x [y0, y1] (arrays) inside a convex quad: the length of each vertical chord, clipped to the box,
    is linear in x between the breakpoints (quad vertices, where an edge crosses y0 or y1, the box's sides), so the
    midpoint rule over those pieces is exact."""
    a, b = quad, np.roll(quad, -1, axis=0)
    brk = [x0, x1] + [np.full_like(x0, vx) for vx in quad[:, 0]]
    for (ax, ay), (bx, by) in zip(a, b):
        if ay != by:
            for yy in (y0, y1):
                brk.append(ax + (yy - ay) * (bx - ax) / (by - ay))
    B = np.sort(np.clip(np.stack(brk, axis=1), x0[:, None], x1[:, None]), axis=1)
    X = 0.5 * (B[:, 1:] + B[:, :-1])
    lo, hi = np.full(X.shape, np.inf), np.full(X.shape, -np.inf)
    for (ax, ay), (bx, by) in zip(a, b):
        if ax == bx:
            continue
        on = (X >= min(ax, bx)) & (X <= max(ax, bx))
        yv = ay + (X - ax) * (by - ay) / (bx - ax)
        lo = np.where(on, np.minimum(lo, yv), lo)
        hi = np.where(on, np.maximum(hi, yv), hi)
    chord = np.maximum(np.minimum(hi, y1[:, None]) - np.maximum(lo, y0[:, None]), 0.0)
    return (chord * np.diff(B, axis=1)).sum(axis=1)


def lens_points(radius, n):
    """Midpoints of n x 2n equal-area cells of the disk (the GPU samples it uniformly)."""
    if radius == 0:
        return np.zeros((1, 2))
    r = radius * np.sqrt((np.arange(n) + 0.5) / n)
    th = 2 * np.pi * (np.arange(2 * n) + 0.5) / (2 * n)
    return np.stack([np.outer(r, np.cos(th)).ravel(), np.outer(r, np.sin(th)).ravel()], axis=1)


def light_share(cam, W, H, n_lens, grow=0.0):
    """p per pixel (H, W): the share of its footprint, grown by `grow` pixels on each side, whose rays hit the light,
    averaged over the lens."""
    quads = [light_quad(cam, W, H, l) for l in lens_points(cam.lens_radius, n_lens)]
    allq = np.concatenate(quads)
    y, x = np.mgrid[0:H, 0:W].astype(np.float64)
    x0, x1, y0, y1 = x.ravel() - grow, x.ravel() + 1 + grow, y.ravel() - grow, y.ravel() + 1 + grow
    near = (x1 >= allq[:, 0].min()) & (x0 <= allq[:, 0].max()) & (y1 >= allq[:, 1].min()) & (y0 <= allq[:, 1].max())
    p = np.zeros(W * H)
    for q in quads:
        p[near] += box_quad_area(q, x0[near], x1[near], y0[near], y1[near])
    return (p / len(quads) / (1 + 2 * grow) ** 2).reshape(H, W)


_CF = {}


def closed_form(vb, aperture):
    """(camera, p, pixels certain to be 0, pixels certain to be 1): certain = the same when the footprint grows by a
    quarter pixel, so no lens point between the quadrature's can change it."""
    if aperture not in _CF:
        cam = cf_camera(vb, aperture)
        n = 64
        p = light_share(cam, CF_W, CF_H, n)
        if aperture:
            p2 = light_share(cam, CF_W, CF_H, int(round(n * np.sqrt(2))))  # twice the points
            assert np.abs(p - p2).max() <= 1e-4, np.abs(p - p2).max()
        g = light_share(cam, CF_W, CF_H, n, grow=0.25)
        _CF[aperture] = (cam, p, g == 0.0, g == 1.0)
    return _CF[aperture]


def check_closed_form(rgb, spp, p, zero, one, label):
    assert np.array_equal(rgb[..., 0], rgb[..., 1]) and np.array_equal(rgb[..., 0], rgb[..., 2]), label
    k = rgb[..., 0].astype(np.float64) * spp / 15.0
    assert np.array_equal(k, np.round(k)), label  # every sample is 0 or 15
    assert (rgb[zero] == 0.0).all() and (rgb[one] == 15.0).all(), (label, rgb[zero].max(), rgb[one].min())
    rest = ~zero & ~one
    np_, var = spp * p[rest], spp * p[rest] * (1 - p[rest])
    dev = np.abs(k[rest] - np_)
    assert (dev <= 4.5 * np.sqrt(var) + 1).all(), (label, np.argwhere(rest)[np.argmax(dev - 4.5 * np.sqrt(var))], dev.max())
    edge = var >= 1.0
    x2 = float((((k[rest] - np_) ** 2)[edge] / var[edge]).sum())
    pval = sst.chi2.sf(x2, int(edge.sum()))
    print(f"{label}: {int(zero.sum())} pixels exactly 0, {int(one.sum())} exactly 15, {int(edge.sum())} edge pixels, "
          f"max |k - np| / sd {(dev[edge] / np.sqrt(var[edge])).max():.2f}, chi-square {x2:.1f} on {int(edge.sum())} (p-value {pval:.3f})")
    assert pval >= 1e-4, (label, x2, int(edge.sum()))
    return int(edge.sum())


@pytest.mark.parametrize("aperture", [0.0, 30.0], ids=["pinhole", "lens"])
def test_closed_form_of_the_generation_stage_on_the_oracle(vb, po, aperture):
    """The closed form is the reference's law too: the oracle (Camera::get_ray with its rejection-sampled disk) meets it."""
    scene, _ = get_scene(vb, "cornell_box")
    cam, p, zero, one = closed_form(vb, aperture)
    assert zero.sum() > 1000 and one.sum() >= (20 if aperture == 0 else 10)
    rgb, _, st = po.OracleScene(scene).render(cam, vb.render_params(CF_W, CF_H, 1024, 1, seed=3))
    assert st.rays == st.paths
    assert check_closed_form(rgb, 1024, p, zero, one, f"oracle {aperture}") >= 30


@gpu
@pytest.mark.parametrize("aperture", [0.0, 30.0], ids=["pinhole", "lens"])
def test_closed_form_of_the_generation_stage(vb, ctx, monkeypatch, aperture):
    scene, _ = get_scene(vb, "cornell_box")
    cam, p, zero, one = closed_form(vb, aperture)
    ctx.upload(scene)
    runs = [("AUTO", 0, None), ("AUTO", vb.VK_FLAG_STRICT_MATH, None), ("AUTO", 0, "VECCHIO_NO_STATIC_FLAT"),
            ("AUTO", 0, "VECCHIO_NO_SIMPLE")]
    runs += [(v, f, None) for v in ("MEGAKERNEL", "WAVEFRONT", "STAGED", "WARPQ") for f in (0, vb.VK_FLAG_STRICT_MATH)]
    for v, f, env in runs:
        if env:
            monkeypatch.setenv(env, "1")
        rgb, _, st = ctx.render(cam, vb.render_params(CF_W, CF_H, CF_SPP, 1, seed=9, variant=getattr(vb, "VK_VARIANT_" + v), flags=f))
        if env:
            monkeypatch.delenv(env)
        assert st.rays == st.paths
        check_closed_form(rgb, CF_SPP, p, zero, one, f"{v} flags {f} {env or ''} aperture {aperture}")
    for v in ("AUTO", "WARPQ", "MEGAKERNEL"):  # a batch: the same camera at seeds 9, 10, 11
        got, st = ctx.render_frames([cam] * 3, vb.render_params(CF_W, CF_H, CF_SPP, 1, seed=9, variant=getattr(vb, "VK_VARIANT_" + v)))
        for f in range(3):
            check_closed_form(got[f], CF_SPP, p, zero, one, f"batch {v} frame {f} aperture {aperture}")
        assert not np.array_equal(got[0], got[1])
