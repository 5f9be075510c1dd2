"""Adaptive sampling of a batch of frames (vk_render_frames_adaptive*) where no GPU is needed: the exports and their
declarations in the header, the ctypes table and the Rust binding, and the checks the Python wrappers make before they
call the library."""
import ctypes
import os
import re

import pytest

from conftest import ROOT

NAMES = ("vk_render_frames_adaptive", "vk_render_frames_adaptive_rgb8")


def test_frames_adaptive_symbols_are_exported_and_declared(vb):
    lib = ctypes.CDLL(vb.gpu_lib()._name)
    hdr = open(os.path.join(ROOT, "include", "vecchio_gpu.h")).read()
    for name in NAMES:
        assert name in vb.GPU_SYMBOLS and hasattr(lib, name)
        assert re.search(r"\bint " + name + r"\(vk_ctx\* ctx, const vk_camera\* cams, uint32_t n_frames,", hdr), name
        assert getattr(vb.gpu_lib(), name).restype is ctypes.c_int
        assert len(getattr(vb.gpu_lib(), name).argtypes) == 9


def test_rust_binding_declares_and_wraps_them():
    src = open(os.path.join(ROOT, "rust", "gpu.rs")).read()
    for name in NAMES:
        assert re.search(r"pub fn " + name + r"\(ctx: \*mut vk_ctx, cams: \*const vk_camera, n_frames: u32,", src), name
    assert "pub fn render_frames_adaptive(" in src and "pub fn render_frames_adaptive_rgb8(" in src


class _NoLibrary:
    """Stands in for the CUDA library: any call through it fails the test."""

    def __getattr__(self, name):
        raise AssertionError(f"{name} was called")


def _offline_context(vb):
    ctx = vb.Context.__new__(vb.Context)  # no device needed: the checks come first
    ctx._L, ctx._h = _NoLibrary(), None
    return ctx


@pytest.mark.parametrize("method", ["render_frames_adaptive", "render_frames_adaptive_rgb8"])
@pytest.mark.parametrize("pass_spp, max_error, match", [(0, 1.0, "pass_spp"), (-3, 1.0, "pass_spp"),
                                                        (16, float("nan"), "max_error"), (16, -0.5, "max_error")])
def test_render_frames_adaptive_rejects_bad_arguments_before_the_library(vb, method, pass_spp, max_error, match):
    cams = [vb._abi.vk_camera(), vb._abi.vk_camera()]
    with pytest.raises(ValueError, match=match):
        getattr(_offline_context(vb), method)(cams, vb.render_params(8, 8, 16), pass_spp, max_error)


@pytest.mark.parametrize("method", ["render_frames_adaptive", "render_frames_adaptive_rgb8"])
def test_render_frames_adaptive_rejects_an_empty_camera_list_before_the_library(vb, method):
    with pytest.raises(ValueError, match="at least one camera"):
        getattr(_offline_context(vb), method)([], vb.render_params(8, 8, 16), 8, 1.0)
