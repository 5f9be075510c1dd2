"""The callers either side of the path (SURVEY 8f rows 2 and 4), host logic only: the output conversion and
P3 writer of src/main.rs:200-214, the frame-loop program's behaviour without a device, and the additive
checkpoint / merge of sample sums.  The oracle stands in for the GPU as the renderer of slices here (same
``render(cam, params, want_sumsq)`` signature, same spp-slice semantics); the GPU versions of these checks are
in test_zz_frames_gpu.py."""
import os
import subprocess

import numpy as np
import pytest

from conftest import HAS_GPU, ROOT, get_scene

RENDER_BIN = os.path.join(ROOT, "vecchio_b200", "lib", "vecchio_gpu_render")


def reference_ppm_text(rgb8):
    """src/main.rs:205-213 restated: header lines, then `writeln!("{} {} {}")` per pixel in file order."""
    h, w, _ = rgb8.shape
    lines = ["P3", f"{w} {h}", "255"] + [f"{r} {g} {b}" for r, g, b in rgb8.reshape(-1, 3).tolist()]
    return "\n".join(lines) + "\n"


def parse_ppm(path):
    tok = open(path).read().split()
    assert tok[0] == "P3" and tok[3] == "255"
    w, h = int(tok[1]), int(tok[2])
    return np.array(tok[4:], dtype=np.int64).reshape(h, w, 3)


def test_frame_to_rgb8_is_to_color_with_rows_flipped(vb, po):
    rng = np.random.default_rng(7)
    f = (rng.random((9, 13, 3), dtype=np.float32) * 1.4).astype(np.float32)
    f[0, 0] = (np.nan, -1.0, np.inf)  # NaN -> 0, sqrt(-1) = NaN -> 0, inf clamps to 0.999 -> 255
    f[1, 1] = (0.0, 0.25, 0.998001)   # 0, 128, 255 (sqrt = 0.999 exactly at the clamp)
    out = vb.frame_to_rgb8(f)
    assert out.dtype == np.uint8 and out.shape == f.shape
    assert (out == vb.to_color(f)[::-1]).all()
    assert list(out[8, 0]) == [0, 0, 255] and list(out[7, 1][:2]) == [0, 128]
    # the oracle's restatement of Vec3::to_color on the same channels
    for y, x in [(0, 0), (1, 1), (4, 5), (8, 12)]:
        assert list(po.kat("to_color", f[y, x], 3)) == list(out[8 - y, x])


@pytest.mark.parametrize("h,w", [(7, 11), (64, 64), (225, 400)])
def test_frame_to_rgb8_vector_and_scalar_paths_agree_with_to_color(vb, h, w):
    """Rows are converted 16 channels at a time with a scalar tail: bin edges ((k/256)^2), NaN, +-inf and negative
    values at every lane position, row lengths that are and are not multiples of 16."""
    rng = np.random.default_rng(h * 1000 + w)
    f = (rng.random((h, w, 3), dtype=np.float32) * 1.5 - 0.1).astype(np.float32)
    for value, share in ((np.nan, 0.02), (np.inf, 0.02), (-np.inf, 0.02)):
        f[rng.random(f.shape) < share] = value
    edges = ((rng.integers(0, 257, f.shape) / 256.0) ** 2).astype(np.float32)
    m = rng.random(f.shape) < 0.3
    f[m] = edges[m]
    m = rng.random(f.shape) < 0.1
    f[m] = np.nextafter(edges[m], np.float32(0))
    assert (vb.frame_to_rgb8(f) == vb.to_color(f)[::-1]).all()


def test_write_ppm_is_byte_for_byte_the_reference_writer(vb, tmp_path):
    rng = np.random.default_rng(3)
    for h, w in [(1, 1), (3, 5), (17, 33), (400, 300)]:  # the last one spans two 1 MiB blocks of text
        rgb8 = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
        rgb8[0, 0] = (0, 9, 10)
        rgb8[-1, -1] = (99, 100, 255)
        p = str(tmp_path / f"f_{h}x{w}.ppm")
        vb.write_ppm(p, rgb8)
        assert open(p).read() == reference_ppm_text(rgb8)
        assert (parse_ppm(p) == rgb8).all()


def test_write_ppm_reports_io_errors(vb, tmp_path):
    with pytest.raises(vb.VecchioError, match="cannot create"):
        vb.write_ppm(str(tmp_path / "no_such_dir" / "x.ppm"), np.zeros((2, 2, 3), np.uint8))


def test_frame_filename(vb):
    assert vb.frame_filename(0) == "output_0000.ppm"  # format!("output_{:04}.ppm") src/main.rs:201
    assert vb.frame_filename(42, "out") == "out/output_0042.ppm"
    assert vb.frame_filename(12345, "out/") == "out/output_12345.ppm"


def test_render_program_usage_and_scene_numbers():
    r = subprocess.run([RENDER_BIN, "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--scene" in r.stdout
    r = subprocess.run([RENDER_BIN, "--scene", "6"], capture_output=True, text=True)  # match arm `_` src/main.rs:166
    assert r.returncode == 2 and "Not a valid scene" in r.stderr
    r = subprocess.run([RENDER_BIN, "--scene", "no_such_scene", "--width", "32", "--spp", "1"], capture_output=True, text=True)
    assert r.returncode == 1 and "Not a valid scene" in r.stderr
    for bad in (["--spp", "0"], ["--width", "1"], ["--gpus", "4", "--spp", "3"], ["--variant", "cpu"], ["--bogus"]):
        assert subprocess.run([RENDER_BIN] + bad, capture_output=True).returncode == 2


@pytest.mark.skipif(HAS_GPU, reason="a GPU is present")
def test_render_program_has_no_cpu_path(tmp_path):
    r = subprocess.run([RENDER_BIN, "--width", "32", "--spp", "2", "--out-dir", str(tmp_path)], capture_output=True,
                       text=True, cwd=ROOT)
    assert r.returncode == 1
    assert "Generating scene..." in r.stderr and "no CPU fallback" in r.stderr
    assert not list(tmp_path.iterdir())


# ---------------------------------------------------------------------------------------------------------
# additive checkpoint / merge

W = H = 24
SPP = 8


@pytest.fixture(scope="module")
def cornell(vb, po):
    scene, cam = get_scene(vb, "cornell_box")
    return po.OracleScene(scene), cam


def params_and_key(vb, cam, **kw):
    from vecchio_b200 import accumulate
    p = vb.render_params(W, H, kw.pop("spp", SPP), 20, seed=kw.pop("seed", 5), **kw)
    return p, accumulate.frame_key("cornell_box", 1, cam, p)


def test_slices_add_up_to_the_frame(vb, cornell):
    from vecchio_b200 import accumulate
    orc, cam = cornell
    p, key = params_and_key(vb, cam)
    full, full_sq, st_full = orc.render(cam, p, want_sumsq=True)
    acc = accumulate.FrameAccumulator(key, with_sumsq=True)
    assert acc.missing() == [(0, SPP)] and not acc.complete
    n = accumulate.render_resumable(orc, cam, p, acc, slice_spp=3)
    assert n == 3 and acc.complete and acc.missing() == [] and acc.samples_done == SPP
    # same Philox samples, only the order of the fp32 additions differs
    assert np.allclose(acc.frame(), full, rtol=2e-6, atol=1e-7)
    assert np.allclose(acc.sumsq, full_sq, rtol=2e-6, atol=1e-7)
    assert acc.paths == st_full.paths == W * H * SPP and acc.rays == st_full.rays
    assert (vb.frame_to_rgb8(acc.frame()).astype(int) - vb.frame_to_rgb8(full).astype(int)).__abs__().max() <= 1


def test_merge_of_checkpoints_from_two_runs(vb, cornell, tmp_path):
    from vecchio_b200 import accumulate
    orc, cam = cornell
    p, key = params_and_key(vb, cam)
    full, _, _ = orc.render(cam, p)
    a, b = accumulate.FrameAccumulator(key), accumulate.FrameAccumulator(key)
    pa, pb = vb.render_params(W, H, SPP, 20, seed=5, spp_begin=5, spp_count=3), vb.render_params(W, H, SPP, 20, seed=5, spp_begin=0, spp_count=5)
    a.add(5, 3, orc.render(cam, pa)[0])
    b.add(0, 5, orc.render(cam, pb)[0])
    assert a.missing() == [(0, 5)] and b.missing() == [(5, 8)]
    fa, fb = str(tmp_path / "a.npz"), str(tmp_path / "b.npz")
    a.save(fa)
    b.save(fb)
    m = accumulate.FrameAccumulator.load(fa)
    assert m.key == key and m.ranges == [(5, 8)] and (m.mean_part == a.mean_part).all()
    m.merge(accumulate.FrameAccumulator.load(fb))
    assert m.complete and np.allclose(m.frame(), full, rtol=2e-6, atol=1e-7)
    # the order of the merge does not show in the fp32 frame
    m2 = accumulate.FrameAccumulator.load(fb)
    m2.merge(accumulate.FrameAccumulator.load(fa))
    assert (m2.frame() == m.frame()).all()


def test_double_counting_and_foreign_frames_are_refused(vb, cornell):
    from vecchio_b200 import accumulate
    orc, cam = cornell
    p, key = params_and_key(vb, cam)
    img = np.zeros((H, W, 3), np.float32)
    a = accumulate.FrameAccumulator(key)
    a.add(0, 4, img)
    with pytest.raises(ValueError, match="already accumulated"):
        a.add(3, 2, img)
    with pytest.raises(ValueError, match="outside"):
        a.add(6, 3, img)
    with pytest.raises(ValueError, match="shape"):
        a.add(4, 1, np.zeros((H, W + 1, 3), np.float32))
    with pytest.raises(ValueError, match="sum-of-squares"):
        a.add(4, 1, img, sumsq=img)
    assert a.ranges == [(0, 4)]  # failed adds leave the total untouched
    b = accumulate.FrameAccumulator(key)
    b.add(2, 4, img)
    with pytest.raises(ValueError, match="already accumulated"):
        a.merge(b)
    for other in (params_and_key(vb, cam, seed=6)[1], params_and_key(vb, cam, flags=1)[1],
                  accumulate.frame_key("cornell_smoke", 1, cam, p), accumulate.frame_key("cornell_box", 2, cam, p)):
        c = accumulate.FrameAccumulator(other)
        c.add(4, 4, img)
        with pytest.raises(ValueError, match="different frames"):
            a.merge(c)
    cam2 = vb.camera_new((278, 278, -700), (278, 278, 0), (0, 1, 0), 40.0, 1.0, 0.0, 10.0, 0.0, 1.0)
    assert accumulate.frame_key("cornell_box", 1, cam2, p) != key
    with pytest.raises(ValueError, match="incomplete"):
        a.frame()
    with pytest.raises(ValueError, match="do not match"):
        accumulate.render_resumable(orc, cam, vb.render_params(W, H, SPP + 1, 20, seed=5), a, 2)


def test_interrupted_render_resumes_from_its_checkpoint(vb, cornell, tmp_path):
    from vecchio_b200 import accumulate
    orc, cam = cornell
    p, key = params_and_key(vb, cam)
    path = str(tmp_path / "frame.npz")
    acc = accumulate.FrameAccumulator(key, with_sumsq=True)
    assert accumulate.render_resumable(orc, cam, p, acc, slice_spp=2, checkpoint_path=path, max_slices=2) == 2
    del acc  # "the process died"
    acc = accumulate.FrameAccumulator.load(path)
    assert acc.ranges == [(0, 4)] and acc.sumsq is not None and acc.paths == W * H * 4
    preview = acc.frame(allow_partial=True)
    half = orc.render(cam, vb.render_params(W, H, 4, 20, seed=5))[0]  # the same 4 samples as a 4-spp frame
    assert np.allclose(preview, half, rtol=2e-6, atol=1e-7)
    assert accumulate.render_resumable(orc, cam, p, acc, slice_spp=3, checkpoint_path=path) == 2  # [4,7) and [7,8)
    assert acc.complete and accumulate.render_resumable(orc, cam, p, acc, slice_spp=3) == 0
    full, full_sq, _ = orc.render(cam, p, want_sumsq=True)
    assert np.allclose(acc.frame(), full, rtol=2e-6, atol=1e-7)
    assert np.allclose(accumulate.FrameAccumulator.load(path).sumsq, full_sq, rtol=2e-6, atol=1e-7)
    assert not [f for f in os.listdir(tmp_path) if ".tmp" in f]


def test_standard_error_from_the_sum_of_squares(vb, cornell):
    from vecchio_b200 import accumulate
    orc, cam = cornell
    p, key = params_and_key(vb, cam)
    acc = accumulate.FrameAccumulator(key, with_sumsq=True)
    samples = []
    for s in range(SPP):  # one-sample slices: slice * spp is the sample itself
        ps = vb.render_params(W, H, SPP, 20, seed=5, spp_begin=s, spp_count=1)
        rgb, sq, st = orc.render(cam, ps, want_sumsq=True)
        acc.add(s, 1, rgb, sq, st)
        samples.append(rgb.astype(np.float64) * SPP)
    samples = np.stack(samples)
    assert acc.dropped_samples == 0
    expect = samples.std(axis=0, ddof=1) / np.sqrt(SPP)
    assert np.allclose(acc.standard_error(), expect, rtol=1e-4, atol=1e-6)
