"""Batches of frames (vk_render_frames*, `vecchio_gpu_render --batch K`) where no GPU is needed: the program's options,
its refusal to run without a device, and the checks the Python wrapper makes before it calls the library."""
import subprocess

import pytest

from conftest import HAS_GPU, ROOT
from test_frames_and_checkpoints import RENDER_BIN


def test_usage_lists_batch():
    r = subprocess.run([RENDER_BIN, "--help"], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0 and "--batch K" in r.stdout


@pytest.mark.parametrize("value", ["0", "x", "-1", ""])
def test_bad_batch_is_a_usage_error(value, tmp_path):
    r = subprocess.run([RENDER_BIN, "--batch", value, "--out-dir", str(tmp_path)], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 2 and "usage:" in r.stderr
    assert not list(tmp_path.iterdir())


def test_batch_without_a_value_is_a_usage_error():
    r = subprocess.run([RENDER_BIN, "--batch"], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 2 and "needs a value" in r.stderr


@pytest.mark.skipif(HAS_GPU, reason="a GPU is present")
def test_batched_program_has_no_cpu_path(tmp_path):
    r = subprocess.run([RENDER_BIN, "--scene", "3", "--width", "32", "--spp", "2", "--batch", "4", "--out-dir", str(tmp_path)],
                       capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 1
    assert "vk_create" in r.stderr and "no CPU fallback" in r.stderr
    assert not list(tmp_path.iterdir())


def test_stress_grid_of_the_gpu_tests_runs_the_dynamic_megakernel(vb):
    # tests/test_zz_batch_frames_gpu.py renders stress_spheres at grid 300 to cover the dynamic lane megakernel's batches
    scene = vb.Scene("stress_spheres", seed=1, param=300)
    assert vb.scene_check(scene.desc_ptr)["dynamic_megakernel"] == 1
    scene.close()


class _NoLibrary:
    """Stands in for the CUDA library: any call through it fails the test."""

    def __getattr__(self, name):
        raise AssertionError(f"{name} was called")


@pytest.mark.parametrize("method", ["render_frames", "render_frames_rgb8"])
def test_render_frames_rejects_an_empty_camera_list_before_the_library(vb, method):
    ctx = vb.Context.__new__(vb.Context)  # no device needed: the check comes first
    ctx._L, ctx._h = _NoLibrary(), None
    with pytest.raises(ValueError, match="at least one camera"):
        getattr(ctx, method)([], vb.render_params(8, 8, 1))
    m = vb.MultiContext.__new__(vb.MultiContext)
    m._L, m._h = _NoLibrary(), None
    with pytest.raises(ValueError, match="at least one camera"):
        m.render_frames_rgb8(iter(()), vb.render_params(8, 8, 1))


def test_batch_symbols_are_exported_and_declared(vb):
    import ctypes
    lib = ctypes.CDLL(vb.gpu_lib()._name)
    for name in ("vk_render_frames", "vk_render_frames_rgb8", "vk_multi_render_frames_rgb8"):
        assert name in vb.GPU_SYMBOLS and hasattr(lib, name)
