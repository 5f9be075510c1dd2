"""Adaptive sampling (vk_render_adaptive*, `vecchio_gpu_render --adaptive E`) where no GPU is needed: the program's options,
its refusal to run without a device, the checks the Python wrapper makes before it calls the library, and the exports."""
import ctypes
import subprocess

import pytest

from conftest import HAS_GPU, ROOT
from test_frames_and_checkpoints import RENDER_BIN


def test_usage_lists_adaptive():
    r = subprocess.run([RENDER_BIN, "--help"], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0 and "--adaptive E" in r.stdout and "--pass-spp M" in r.stdout
    assert "biased" in r.stdout


@pytest.mark.parametrize("args", [["--adaptive", "-1"], ["--adaptive", "x"], ["--adaptive", ""], ["--adaptive", "nan"],
                                  ["--adaptive", "inf"], ["--adaptive", "1", "--pass-spp", "0"],
                                  ["--adaptive", "1", "--pass-spp", "x"], ["--pass-spp", "16"],
                                  ["--adaptive", "1", "--batch", "2"], ["--adaptive", "1", "--gpus", "2"],
                                  ["--adaptive", "1", "--devices", "0,1"]])
def test_bad_adaptive_options_are_usage_errors(args, tmp_path):
    r = subprocess.run([RENDER_BIN, *args, "--scene", "3", "--width", "32", "--spp", "4", "--out-dir", str(tmp_path)],
                       capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 2 and "usage:" in r.stderr
    assert not list(tmp_path.iterdir())


@pytest.mark.parametrize("option", ["--adaptive", "--pass-spp"])
def test_adaptive_option_without_a_value_is_a_usage_error(option):
    r = subprocess.run([RENDER_BIN, option], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 2 and "needs a value" in r.stderr


@pytest.mark.skipif(HAS_GPU, reason="a GPU is present")
def test_adaptive_program_has_no_cpu_path(tmp_path):
    r = subprocess.run([RENDER_BIN, "--scene", "3", "--width", "32", "--spp", "8", "--adaptive", "2", "--pass-spp", "4",
                        "--out-dir", str(tmp_path)], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 1
    assert "vk_create" in r.stderr and "no CPU fallback" in r.stderr
    assert not list(tmp_path.iterdir())


class _NoLibrary:
    """Stands in for the CUDA library: any call through it fails the test."""

    def __getattr__(self, name):
        raise AssertionError(f"{name} was called")


@pytest.mark.parametrize("method", ["render_adaptive", "render_adaptive_rgb8"])
@pytest.mark.parametrize("pass_spp, max_error, match", [(0, 1.0, "pass_spp"), (-3, 1.0, "pass_spp"),
                                                        (16, float("nan"), "max_error"), (16, -0.5, "max_error")])
def test_render_adaptive_rejects_bad_arguments_before_the_library(vb, method, pass_spp, max_error, match):
    ctx = vb.Context.__new__(vb.Context)  # no device needed: the check comes first
    ctx._L, ctx._h = _NoLibrary(), None
    with pytest.raises(ValueError, match=match):
        getattr(ctx, method)(vb._abi.vk_camera(), vb.render_params(8, 8, 16), pass_spp, max_error)


def test_adaptive_symbols_are_exported_and_declared(vb):
    lib = ctypes.CDLL(vb.gpu_lib()._name)
    for name in ("vk_render_adaptive", "vk_render_adaptive_rgb8"):
        assert name in vb.GPU_SYMBOLS and hasattr(lib, name)
