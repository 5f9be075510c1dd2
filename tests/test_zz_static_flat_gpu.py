"""The warp-queue kernel compiled for cornell_box's flat-program shape (trace_flat_static) against the generic kernel
(VECCHIO_NO_STATIC_FLAT=1): the same entries in the same order with the same arithmetic, so the same frame bit for bit
(integer accumulators: the frame does not depend on scheduling)."""
import numpy as np
import pytest

import vecchio_b200 as vb
from conftest import get_scene


@pytest.mark.gpu
def test_static_shape_kernel_renders_the_generic_kernels_frame(ctx, monkeypatch):
    s, cam = get_scene(vb, "cornell_box")
    assert vb.scene_check(s.desc_ptr)["flat_shape"] != 0
    ctx.upload(s)
    p = vb.render_params(96, 96, 24, 100, seed=5, variant=vb.VK_VARIANT_WARPQ)
    a, qa, sa = ctx.render(cam, p, want_sumsq=True)
    monkeypatch.setenv("VECCHIO_NO_STATIC_FLAT", "1")
    b, qb, sb = ctx.render(cam, p, want_sumsq=True)
    assert a.tobytes() == b.tobytes() and np.array_equal(qa, qb)
    assert (sa.paths, sa.rays, sa.dropped_samples) == (sb.paths, sb.rays, sb.dropped_samples)
