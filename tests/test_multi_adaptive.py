"""Adaptive sampling split over shards of pixels (vk_adaptive_begin_shard, vk_multi_adaptive_*, vk_multi_render_*adaptive_rgb8)
where no GPU is needed: the exports and their declarations, the Rust binding's arity, the checks the Python wrappers make
before they call the library, the shard in a checkpoint's identity, and the claim itself on the host model: for any
tightening sequence of targets the shards' states add up, bit for bit, to the unsharded state."""
import ctypes
import os
import re

import numpy as np
import pytest

import adaptive_model as am
import shard_model as sm
from conftest import ROOT
from test_abi_layouts import _rust_layout, c_layout  # noqa: F401  (the module's gcc layout fixture)

NAMES = ("vk_adaptive_begin_shard", "vk_multi_adaptive_begin", "vk_multi_adaptive_refine", "vk_multi_adaptive_read",
         "vk_multi_adaptive_read_rgb8", "vk_multi_adaptive_export", "vk_multi_adaptive_import", "vk_multi_adaptive_variant",
         "vk_multi_adaptive_destroy", "vk_multi_render_adaptive_rgb8", "vk_multi_render_frames_adaptive_rgb8")


def test_shard_and_multi_symbols_are_exported_and_declared(vb):
    lib = ctypes.CDLL(vb.gpu_lib()._name)
    hdr = open(os.path.join(ROOT, "include", "vecchio_gpu.h")).read()
    for name in NAMES:
        assert name in vb.GPU_SYMBOLS and hasattr(lib, name), name
        assert re.search(r"\b(int|void|uint32_t) " + name + r"\(", hdr), name
    assert re.search(r"#define VK_SHARD_RUN 32\b", hdr)


def test_ctypes_declares_the_multi_calls_like_their_one_gpu_twins(vb):
    L = vb.gpu_lib()
    for f in ("begin", "refine", "read", "read_rgb8", "export", "import", "variant", "destroy"):
        a, b = getattr(L, "vk_multi_adaptive_" + f), getattr(L, "vk_adaptive_" + f)
        assert a.argtypes == b.argtypes and a.restype == b.restype, f
    assert len(L.vk_adaptive_begin_shard.argtypes) == len(L.vk_adaptive_begin.argtypes) + 2


def test_rust_binding_declares_them_with_the_header_s_arity(c_layout):  # noqa: F811
    _, c_protos = c_layout
    _, protos = _rust_layout()
    for name in NAMES:
        assert protos.get(name) == c_protos[name], name
    src = open(os.path.join(ROOT, "rust", "gpu.rs")).read()
    multi = src[src.index("impl MultiGpu {"):]
    for fn in ("pub fn adaptive_session(", "pub fn render_adaptive_rgb8(", "pub fn render_frames_adaptive_rgb8("):
        assert fn in multi, fn
    assert "impl<'a> Drop for MultiAdaptiveSession<'a>" in src


class _NoLibrary:
    """Stands in for the CUDA library: any call through it fails the test."""

    def __getattr__(self, name):
        raise AssertionError(f"{name} was called")


def _offline(vb, cls):
    obj = cls.__new__(cls)
    obj._L, obj._h = _NoLibrary(), None
    return obj


@pytest.mark.parametrize("shard", [(2, 2), (0, 0), (-1, 2), (3, 1)])
def test_a_shard_outside_its_count_is_refused_before_the_library(vb, shard):
    ctx = _offline(vb, vb.Context)
    with pytest.raises(ValueError, match="shard"):
        ctx.adaptive_session([vb._abi.vk_camera()], vb.render_params(8, 8, 16), 8, shard=shard)


@pytest.mark.parametrize("kw, match", [(dict(pass_spp=0, max_error=1.0), "pass_spp"), (dict(pass_spp=8, max_error=-1.0), "max_error"),
                                       (dict(pass_spp=8, max_error=float("nan")), "max_error")])
def test_multi_one_shot_calls_refuse_bad_arguments_before_the_library(vb, kw, match):
    m = _offline(vb, vb.MultiContext)
    cam, p = vb._abi.vk_camera(), vb.render_params(8, 8, 16)
    with pytest.raises(ValueError, match=match):
        m.render_adaptive_rgb8(cam, p, **kw)
    with pytest.raises(ValueError, match=match):
        m.render_frames_adaptive_rgb8([cam, cam], p, **kw)
    with pytest.raises(ValueError, match="camera"):
        m.render_frames_adaptive_rgb8([], p, 8, 1.0)


def test_multi_session_calls_the_multi_api(vb):
    m = _offline(vb, vb.MultiContext)
    with pytest.raises(AssertionError, match="vk_multi_adaptive_begin was called"):
        m.adaptive_session([vb._abi.vk_camera()], vb.render_params(8, 8, 16), 8)


def _cams(vb, n=2):
    cs = []
    for i in range(n):
        c = vb._abi.vk_camera()
        c.origin[0] = float(i)
        cs.append(c)
    return cs


def _session(vb, shard=None):
    s = vb.AdaptiveSession.__new__(vb.AdaptiveSession)
    s._L, s._h, s._ctx = _NoLibrary(), None, None
    s.cams, s.params = _cams(vb), vb.render_params(4, 3, 40)
    s.pass_spp, s.n_frames, s.single, s.reached, s.variant = 8, 2, False, None, vb.VK_VARIANT_WARPQ
    if shard is not None:
        s.shard = shard
    return s


def test_a_shard_s_key_names_the_shard_and_a_whole_session_s_key_is_unchanged(vb):
    from vecchio_b200.adaptive_checkpoint import session_key
    whole = _session(vb).key("cornell_box", 1)
    assert "shard" not in whole
    assert whole == session_key("cornell_box", 1, _cams(vb), vb.render_params(4, 3, 40), 8, vb.VK_VARIANT_WARPQ)
    part = _session(vb, (1, 3)).key("cornell_box", 1)
    assert part == dict(whole, shard=[1, 3])


@pytest.mark.parametrize("writer, reader", [((1, 3), None), (None, (1, 3)), ((1, 3), (2, 3)), ((1, 3), (1, 4))])
def test_a_shard_checkpoint_never_loads_into_another_session(vb, tmp_path, writer, reader):
    from vecchio_b200.adaptive_checkpoint import save_state
    w = _session(vb, writer)
    key = w.key("cornell_box", 1)
    path = str(tmp_path / "s.npz")
    z = np.zeros((2, 3, 4, 3), dtype=np.int64)
    save_state(path, key, z, z.astype(np.uint64), np.zeros((2, 3, 4), dtype=np.uint32), None)
    with pytest.raises(ValueError, match="not this session's identity"):
        _session(vb, reader).load(path, key)
    with pytest.raises(ValueError, match="another session"):
        _session(vb, reader).load(path, _session(vb, reader).key("cornell_box", 1))
    with pytest.raises(AssertionError, match="vk_adaptive_import was called"):
        _session(vb, writer).load(path, key)  # (its own identity reaches the library)


# ---- the claim on the host model ----

def _streams(rng, shape, cap):
    """Per pixel, `cap` random samples of three channels as fixed-point sum units and their squares, each pixel with its
    own mean and noise so that the rule stops pixels at many different counts; returns states[b] = (sums, squares) after
    samples [0, b) for every b <= cap."""
    mean = rng.uniform(0.05, 0.9, size=shape + (1, 3))
    sigma = np.exp(rng.uniform(np.log(0.002), np.log(0.5), size=shape + (1, 1)))
    x = np.clip(mean + sigma * rng.standard_normal(size=shape + (cap, 3)), 0.0, 4.0)
    units = np.rint(x * am.ACC_UNITS).astype(np.int64)
    sq = ((units.astype(object) ** 2) >> 28).astype(np.uint64)  # (about square_units; any fixed integers will do here)
    cs = np.concatenate([np.zeros(shape + (1, 3), np.int64), np.cumsum(units, axis=-2)], axis=-2)
    cq = np.concatenate([np.zeros(shape + (1, 3), np.uint64), np.cumsum(sq, axis=-2, dtype=np.uint64)], axis=-2)
    return {b: (cs[..., b, :], cq[..., b, :]) for b in range(cap + 1)}


SEQUENCES = {
    "error 8-4-2": [(64, 0, 8.0), (64, 0, 4.0), (64, 0, 2.0)],
    "min_spp rise": [(64, 0, 4.0), (64, 24, 4.0), (64, 40, 4.0)],
    "cap raise": [(24, 0, 3.0), (48, 0, 3.0), (64, 0, 2.0)],
}


@pytest.mark.parametrize("seq", list(SEQUENCES))
@pytest.mark.parametrize("k", [1, 3])
def test_shard_states_add_up_to_the_whole_state(k, seq):
    rng = np.random.default_rng(k * 100 + len(seq))
    shape = (k, 5, 7) if k > 1 else (5, 7)  # W*H = 35: not a multiple of 32
    M = 8
    states = _streams(rng, shape, 64)
    n_pix = int(np.prod(shape))
    runs = -(-n_pix // sm.SHARD_RUN)
    whole = None
    for t in SEQUENCES[seq]:
        whole = am.predict(states, t, M, start=whole)
    assert len(np.unique(whole[0])) >= 3  # the rule stopped pixels at several counts
    for n_shards in (1, 2, 3, 8, runs + 2):  # (runs + 2: shards that own no pixel)
        parts = []
        for sh in range(n_shards):
            part = None
            for t in SEQUENCES[seq]:
                part = sm.predict_shard(states, t, M, (sh, n_shards), start=part)
            mine = sm.owned(shape, sh, n_shards)
            assert not part[0][~mine].any() and not part[1][~mine].any() and not part[2][~mine].any()
            parts.append(part)
        for i, dt in enumerate((np.uint32, np.int64, np.uint64)):
            total = np.zeros_like(whole[i])
            for part in parts:
                total = total + part[i]
            assert total.dtype == whole[i].dtype == dt and np.array_equal(total, whole[i]), (n_shards, i)
        assert sum(int(p[0].astype(np.int64).sum()) for p in parts) == int(whole[0].astype(np.int64).sum())  # paths


@pytest.mark.parametrize("shape", [(5, 7), (3, 5, 7), (2, 32, 3), (1,)])
@pytest.mark.parametrize("n_shards", [1, 2, 3, 8, 40])
def test_the_shards_partition_the_pixels_in_runs_of_32(shape, n_shards):
    own = np.stack([sm.owned(shape, k, n_shards) for k in range(n_shards)])
    assert (own.sum(axis=0) == 1).all()
    flat = own.reshape(n_shards, -1)
    for k in range(n_shards):
        g = np.flatnonzero(flat[k])
        assert ((g // 32) % n_shards == k).all()
        runs = -(-flat.shape[1] // 32)
        want = sum(min(32, flat.shape[1] - 32 * r) for r in range(k, runs, n_shards))  # vk_api.cu's shard_pixels
        assert len(g) == want
