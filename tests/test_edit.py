"""Node edits on the host side (no GPU): HostScene.place_node gives the flat description of the scene file edited the same way,
array for array, and refuses bad arguments without changing it.  The GPU side is tests/test_gpu_edit.py."""
import ctypes as C

import numpy as np
import pytest

import chess2rt_b200 as c2
from chess2rt_b200 import api
from sdl_edit import SC, assert_same_desc, desc_arrays, load_edited

CHESS = f"{SC}/chessboard.sdl"
LECTURE5 = f"{SC}/lecture5.sdl"

CASES = [
    ("chess_move", CHESS, [("e2", dict(translate=(10.0, 0.0, -10.0)))]),
    ("chess_capture", CHESS, [("d7", dict(translate=(130.0, 0.0, 40.0)))]),
    ("chess_promotion", CHESS, [("a7", dict(geometry="queen", translate=(-70.0, 0.0, 70.0)))]),
    ("chess_bishop_unscaled", CHESS, [("c1", dict(translate=(-30.0, 0.0, -70.0)))]),
    ("chess_two_edits", CHESS, [("e2", dict(translate=(10.0, 0.0, -10.0))), ("e7", dict(translate=(10.0, 0.0, 10.0)))]),
    ("lecture5_rotate", LECTURE5, [("globe", dict(rotate=(1.5, 0.5, 2.0)))]),
    ("lecture5_scale_rotate_translate", LECTURE5, [("S2", dict(scale=(2.0, 1.0, 1.0), rotate=(1.0, 3.0, 1.0),
                                                                translate=(90.0, 20.0, 200.0)))]),
]


@pytest.mark.parametrize("name,path,edits", CASES, ids=[c[0] for c in CASES])
def test_place_node_matches_the_edited_scene_file(tmp_path, name, path, edits):
    s = c2.HostScene(path)
    desc_arrays(s)   # the flat description exists before the edit: it is updated in place
    for node, kw in edits:
        s.place_node(node, **kw)
    ref = load_edited(str(tmp_path), path, edits)
    assert_same_desc(desc_arrays(s), desc_arrays(ref))
    # and the same when the description is first built after the edit
    s2 = c2.HostScene(path)
    for node, kw in edits:
        s2.place_node(s2.node_index(node), **kw)
    assert_same_desc(desc_arrays(s2), desc_arrays(ref))


def test_place_node_edits_change_only_the_edited_node(tmp_path):
    s = c2.HostScene(CHESS)
    before = desc_arrays(s)
    i = s.node_index("e2")
    s.place_node("e2", translate=(10.0, 0.0, -10.0))
    after = desc_arrays(s)
    for k in before:
        if k != "node_offset":
            assert before[k].tobytes() == after[k].tobytes(), k
    changed = np.flatnonzero(before["node_offset"] != after["node_offset"]) // 3
    assert set(changed) == {i}
    assert tuple(after["node_offset"][3 * i:3 * i + 3]) == (10.0, 0.0, -10.0)


def test_place_node_refuses_bad_arguments_and_changes_nothing():
    s = c2.HostScene(CHESS)
    before = desc_arrays(s)
    n = s.info()["nodes"]
    for bad in (n, -1, 10 ** 6):
        with pytest.raises(c2.C2rtError, match="out of range") as e:
            s.place_node(bad, translate=(0, 0, 0))
        assert e.value.status == -1
    with pytest.raises(KeyError):
        s.place_node("z9", translate=(0, 0, 0))
    with pytest.raises(c2.C2rtError, match="no geometry named") as e:
        s.place_node("a2", geometry="dragon", translate=(0, 0, 0))
    assert e.value.status == -1
    with pytest.raises(ValueError):
        s.place_node("a2", translate=(0, 0))
    assert_same_desc(desc_arrays(s), before)


def test_set_nodes_refuses_a_null_scene_before_any_device():
    m = np.eye(3).reshape(-1)
    off = np.zeros(3)
    node = np.zeros(1, np.uint32)
    geom = np.zeros(1, np.int32)
    rc = api.lib.c2rt_scene_set_nodes(None, 1, node.ctypes.data, geom.ctypes.data, m.ctypes.data, m.ctypes.data,
                                      m.ctypes.data, off.ctypes.data)
    assert rc == -1 and b"scene is null" in api.lib.c2rt_last_error()
    with pytest.raises(c2.C2rtError, match="scene is null"):
        c2.scene_set_nodes(None, [0], geom=[0])


def test_set_nodes_binding_follows_the_header():
    assert "c2rt_scene_set_nodes" in api.C_ABI_SYMBOLS
    f = api.lib.c2rt_scene_set_nodes
    assert f.argtypes[1] is C.c_size_t and len(f.argtypes) == 8
