"""The flat program's compiled shape (FlatShape, vk_internal.h): vk_scene_upload runs the warp-queue kernel compiled for
the program's shape when it has one, the generic kernel otherwise.  The matcher runs on the host (vk_scene_check)."""
import ctypes as C

import pytest

from conftest import get_scene


def _ref(t, i):
    return (t << 28) | i


def test_cornell_box_has_the_compiled_shape(vb):
    assert vb.scene_check(get_scene(vb, "cornell_box")[0].desc_ptr)["flat_shape"] == 1  # VKF_SHAPE_CORNELL


@pytest.mark.parametrize("name", ["cornell_smoke", "furnace_demo", "balls_demo", "perlin_demo", "random_spheres_demo"])
def test_other_scenes_take_the_generic_kernel(vb, name):
    assert vb.scene_check(get_scene(vb, name)[0].desc_ptr)["flat_shape"] == 0


def test_one_more_rect_is_not_the_cornell_shape(vb):
    """cornell_box with one more wall: a new root over the old one and a copy of rect 0 -- a flat program of the same
    frames but seven world rects, which the Cornell kernel would not test."""
    from vecchio_b200 import _abi

    d = get_scene(vb, "cornell_box")[0].desc
    rects = (_abi.vk_rect * (d.n_rects + 1))(*[d.rects[i] for i in range(d.n_rects)], d.rects[0])
    nodes = (_abi.vk_node * (d.n_nodes + 1))(*[d.nodes[i] for i in range(d.n_nodes)])
    old_root = d.nodes[d.root & 0x0FFFFFFF]
    top = nodes[d.n_nodes]
    for k in range(3):
        top.bb_min[k] = old_root.bb_min[k]
        top.bb_max[k] = old_root.bb_max[k]
    top.left = d.root
    top.right = _ref(_abi.VK_T_RECT, d.n_rects)
    e = _abi.vk_scene_desc()
    C.pointer(e)[0] = d  # (a copy of the description; the arrays below replace two of its pointers)
    e.rects, e.n_rects = C.cast(rects, C.POINTER(_abi.vk_rect)), d.n_rects + 1
    e.nodes, e.n_nodes = C.cast(nodes, C.POINTER(_abi.vk_node)), d.n_nodes + 1
    e.root = _ref(_abi.VK_T_NODE, d.n_nodes)
    info = vb.scene_check(C.pointer(e))
    base = vb.scene_check(get_scene(vb, "cornell_box")[0].desc_ptr)
    assert info["flat_entries"] == base["flat_entries"] + 1 and info["flat_segments"] == base["flat_segments"]
    assert info["flat_shape"] == 0
