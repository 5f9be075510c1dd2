"""Adaptive render sessions (vk_adaptive_*) where no GPU is needed: the exports and their declarations, the Rust binding's
arity and target layout, the checks the Python wrappers make before they call the library, and the checkpoint format."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from test_abi_layouts import _rust_layout, c_layout  # noqa: F401  (the module's gcc layout fixture)

NAMES = ("vk_adaptive_begin", "vk_adaptive_refine", "vk_adaptive_read", "vk_adaptive_read_rgb8", "vk_adaptive_export",
         "vk_adaptive_import", "vk_adaptive_variant", "vk_adaptive_destroy")


def test_session_symbols_are_exported_and_declared(vb):
    lib = ctypes.CDLL(vb.gpu_lib()._name)
    hdr = open(os.path.join(ROOT, "include", "vecchio_gpu.h")).read()
    for name in NAMES:
        assert name in vb.GPU_SYMBOLS and hasattr(lib, name), name
        assert re.search(r"\b(int|void|uint32_t) " + name + r"\(", hdr), name


def test_rust_binding_declares_them_with_the_header_s_arity_and_target_layout(c_layout):  # noqa: F811
    layout, c_protos = c_layout
    structs, protos = _rust_layout()
    for name in NAMES:
        assert protos.get(name) == c_protos[name], name
    want, got = layout["vk_adaptive_target"], structs["vk_adaptive_target"]
    assert got["size"] == want["size"] == 12
    assert [(n, o, s) for n, o, s in got["fields"]] == want["fields"]
    src = open(os.path.join(ROOT, "rust", "gpu.rs")).read()
    for fn in ("pub fn adaptive_session(", "pub fn refine(", "pub fn read(", "pub fn read_rgb8(", "pub fn export(", "pub fn import("):
        assert fn in src, fn
    assert "impl<'a> Drop for AdaptiveSession<'a>" in src


def test_ctypes_target_has_gcc_s_layout(vb, c_layout):  # noqa: F811
    layout, _ = c_layout
    T = vb._abi.vk_adaptive_target
    assert ctypes.sizeof(T) == layout["vk_adaptive_target"]["size"]
    assert [(n, getattr(T, n).offset, getattr(T, n).size) for n, _ in T._fields_] == layout["vk_adaptive_target"]["fields"]


class _NoLibrary:
    """Stands in for the CUDA library: any call through it fails the test."""

    def __getattr__(self, name):
        raise AssertionError(f"{name} was called")


def _offline_session(vb, spp=256, pass_spp=32, reached=None, k=1):
    s = vb.AdaptiveSession.__new__(vb.AdaptiveSession)
    s._L, s._h, s._ctx = _NoLibrary(), None, None
    s.params = vb.render_params(8, 8, spp)
    s.pass_spp, s.n_frames, s.single, s.reached = pass_spp, k, k == 1, reached
    return s


@pytest.mark.parametrize("cams", [[], None])
def test_a_session_needs_cameras_before_the_library(vb, cams):
    ctx = vb.Context.__new__(vb.Context)
    ctx._L, ctx._h = _NoLibrary(), None
    with pytest.raises((ValueError, TypeError)):
        vb.AdaptiveSession(ctx, cams, vb.render_params(8, 8, 16), 8)


def test_a_session_needs_pass_spp(vb):
    ctx = vb.Context.__new__(vb.Context)
    ctx._L, ctx._h = _NoLibrary(), None
    with pytest.raises(ValueError, match="pass_spp"):
        vb.AdaptiveSession(ctx, [vb._abi.vk_camera()], vb.render_params(8, 8, 16), 0)


@pytest.mark.parametrize("reached, kw, match", [
    (None, dict(max_error=float("nan")), "max_error"),
    (None, dict(max_error=-1.0), "max_error"),
    (None, dict(max_error=1.0, spp=0), "spp"),
    (None, dict(max_error=1.0, spp=257), "limit"),
    (None, dict(max_error=1.0, min_spp=-1), "min_spp"),
    ((128, 0, 4.0), dict(max_error=8.0, spp=128), "loosens"),
    ((128, 0, 0.0), dict(max_error=1.0, spp=128), "loosens"),
    ((128, 64, 4.0), dict(max_error=4.0, spp=128, min_spp=32), "min_spp"),
    ((128, 0, 4.0), dict(max_error=4.0, spp=96), "spp"),
    ((100, 0, 4.0), dict(max_error=4.0, spp=128), "pass grid"),
])
def test_refine_refuses_loosening_and_bad_targets_before_the_library(vb, reached, kw, match):
    s = _offline_session(vb, reached=reached)
    with pytest.raises(ValueError, match=match):
        s.refine(**kw)


def _state(rng, k=2, h=3, w=4, pass_spp=8, cap=40):
    counts = rng.choice([8, 16, 24, 32, 40], size=(k, h, w)).astype(np.uint32)
    sums = rng.integers(0, 2 ** 40, size=(k, h, w, 3), dtype=np.int64)
    squares = rng.integers(0, 2 ** 60, size=(k, h, w, 3), dtype=np.uint64)
    return sums, squares, counts, (cap, 0, np.float32(1.5).item())


def _key(vb, seed=1, cams=2):
    from vecchio_b200.adaptive_checkpoint import session_key
    cs = []
    for i in range(cams):
        c = vb._abi.vk_camera()
        c.origin[0] = float(i)
        cs.append(c)
    return session_key("cornell_box", seed, cs, vb.render_params(4, 3, 40), 8, vb.VK_VARIANT_WARPQ)


def test_checkpoint_round_trips(vb, tmp_path):
    from vecchio_b200.adaptive_checkpoint import load_state, save_state
    state = _state(np.random.default_rng(0))
    path = str(tmp_path / "s.npz")
    save_state(path, _key(vb), *state)
    got = load_state(path, _key(vb))
    for a, b in zip(got[:3], state[:3]):
        assert a.dtype == b.dtype and np.array_equal(a, b)
    assert got[3] == state[3]
    save_state(path, _key(vb), state[0] * 0, state[1] * 0, state[2] * 0, None)
    assert load_state(path, _key(vb))[3] is None


@pytest.mark.parametrize("other", [dict(seed=2), dict(cams=3)])
def test_checkpoint_refuses_a_foreign_identity(vb, tmp_path, other):
    from vecchio_b200.adaptive_checkpoint import load_state, save_state
    path = str(tmp_path / "s.npz")
    save_state(path, _key(vb), *_state(np.random.default_rng(1)))
    with pytest.raises(ValueError, match="another session"):
        load_state(path, _key(vb, **other))


def test_key_hashes_every_camera_and_records_the_pass_grid_and_kernel(vb):
    k = _key(vb, cams=2)
    assert len(k["camera"]) == 2 and k["camera"][0] != k["camera"][1]
    assert k["pass_spp"] == 8 and k["variant"] == vb.VK_VARIANT_WARPQ and k["spp"] == 40


def test_an_interrupted_save_leaves_the_previous_checkpoint(vb, tmp_path, monkeypatch):
    from vecchio_b200 import adaptive_checkpoint as ac
    path = str(tmp_path / "s.npz")
    first = _state(np.random.default_rng(2))
    ac.save_state(path, _key(vb), *first)

    def dies(f, **arrays):
        f.write(b"partial")
        raise KeyboardInterrupt

    monkeypatch.setattr(ac.np, "savez", dies)
    with pytest.raises(KeyboardInterrupt):
        ac.save_state(path, _key(vb), *_state(np.random.default_rng(3)))
    monkeypatch.undo()
    got = ac.load_state(path, _key(vb))
    assert all(np.array_equal(a, b) for a, b in zip(got[:3], first[:3]))
    assert os.listdir(tmp_path) == ["s.npz"]


class _FakeSession:
    """What render_adaptive_resumable drives, without a device: records the refines and saves."""

    def __init__(self, vb):
        self.vb, self.reached, self.log = vb, None, []
        self.params = vb.render_params(4, 3, 64)

    def target(self, max_error, spp=None, min_spp=0):
        return self.vb._adaptive_target(max_error, 64 if spp is None else spp, min_spp)

    def refine(self, max_error, spp=None, min_spp=0):
        self.reached = self.target(max_error, spp, min_spp)
        self.log.append(("refine", self.reached))

    def save(self, path, key):
        self.log.append(("save", self.reached))
        open(path, "w").write(repr(self.reached))

    def load(self, path, key):
        self.reached = eval(open(path).read())
        self.log.append(("load", self.reached))


def test_resumable_refines_saves_after_each_target_and_resumes_after_the_reached_one(vb, tmp_path):
    from vecchio_b200.adaptive_checkpoint import render_adaptive_resumable
    path = str(tmp_path / "s.ckpt")
    targets = [(8.0,), (4.0,), (2.0, 64, 16)]
    s = _FakeSession(vb)
    assert render_adaptive_resumable(s, targets[:2], path, key={}) == 2
    assert [e[0] for e in s.log] == ["refine", "save", "refine", "save"]
    s2 = _FakeSession(vb)
    assert render_adaptive_resumable(s2, targets, path, key={}) == 1
    assert s2.log == [("load", (64, 0, 4.0)), ("refine", (64, 16, 2.0)), ("save", (64, 16, 2.0))]


def _offline_with_identity(vb, seed=1, cam_x=0.0, pass_spp=8, variant=None, flags=0, depth=100):
    s = _offline_session(vb, spp=40, pass_spp=pass_spp, k=2)
    cams = []
    for i in range(2):
        c = vb._abi.vk_camera()
        c.origin[0] = float(i) + cam_x
        cams.append(c)
    s.cams = cams
    s.params = vb.render_params(4, 3, 40, max_depth=depth, seed=seed, flags=flags)
    s.variant = vb.VK_VARIANT_WARPQ if variant is None else variant
    return s


@pytest.mark.parametrize("other", [dict(seed=2), dict(cam_x=0.5), dict(pass_spp=16), dict(variant=1), dict(flags=1),
                                   dict(depth=30)])
def test_load_refuses_another_session_s_checkpoint_even_with_its_own_key(vb, tmp_path, other):
    from vecchio_b200.adaptive_checkpoint import save_state
    writer = _offline_with_identity(vb)
    key = writer.key("cornell_box", 1)
    path = str(tmp_path / "s.npz")
    save_state(path, key, *_state(np.random.default_rng(4), k=2, h=3, w=4))
    reader = _offline_with_identity(vb, **other)
    with pytest.raises(ValueError, match="not this session's identity"):
        reader.load(path, key)  # (the library is never called: _NoLibrary would fail the test)
    with pytest.raises(ValueError, match="not this session's identity"):
        reader.save(path, key)


def test_load_with_the_session_s_own_key_reaches_the_import(vb, tmp_path):
    from vecchio_b200.adaptive_checkpoint import save_state
    s = _offline_with_identity(vb)
    key = s.key("cornell_box", 1)
    path = str(tmp_path / "s.npz")
    save_state(path, key, *_state(np.random.default_rng(5), k=2, h=3, w=4))
    with pytest.raises(AssertionError, match="vk_adaptive_import was called"):
        s.load(path, key)
