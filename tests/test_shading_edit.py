"""Shading and light edits on the host side (no GPU): HostScene.set_node_shader / set_shader / set_texture / set_light give the
flat description of the scene file edited the same way, array for array and bit for bit, and refuse bad arguments without
changing it.  The GPU side is tests/test_gpu_shading_edit.py."""
import ctypes as C

import numpy as np
import pytest

import chess2rt_b200 as c2
from chess2rt_b200 import api
from sdl_edit import SC, TSC, assert_same_desc, desc_arrays
from sdl_shading import add_entity, apply_edit, edit_text, load_text, read

CHESS = f"{SC}/chessboard.sdl"
LECTURE5 = f"{SC}/lecture5.sdl"
PROC = f"{SC}/lecture4-proc-texture.sdl"
ZAPHOD = f"{SC}/zaphod.sdl"
HIGHLIGHT = 'Phong "highlight" { color 0.25 0.875 0.25; exponent 20 }'

# (id, scene, spare shader or None, [edits]); an edit is (section, entity, keys) as sdl_shading.apply_edit takes it
CASES = [
    ("chess_highlight", CHESS, HIGHLIGHT, [("Nodes", "e2", dict(shader="highlight"))]),
    ("chess_piece_colour", CHESS, None, [("Shaders", "white_piece", dict(color=(0.875, 0.5, 0.25)))]),
    ("chess_clamps", CHESS, None, [("Shaders", "white_piece", dict(exponent=1e9, strength=-2.0)),
                                   ("Shaders", "black_piece", dict(exponent=1e-9, strength=3e6))]),
    ("chess_phong_to_lambert", CHESS, None, [("Shaders", "white_piece", dict(kind="Lambert", color=(0.5, 0.5, 0.75)))]),
    ("chess_lambert_to_phong", CHESS, None, [("Shaders", "floor_shader", dict(kind="Phong", texture="board", exponent=30.0))]),
    ("chess_drop_texture", CHESS, None, [("Shaders", "floor_shader", dict(texture=None))]),
    ("chess_checker", CHESS, None, [("Textures", "board", dict(color1=(0.5, 0.125, 0.0), color2=(1.0, 1.0, 0.75), size=12.5))]),
    ("lecture5_relight", LECTURE5, None, [("Lights", "light1", dict(pos=(-200.0, 500.0, 100.0), color=(1.0, 0.75, 0.5), power=6e5))]),
    ("lecture5_bitmap_switch", LECTURE5, None, [("Shaders", "csg_shader", dict(texture="world"))]),
    ("proc_frequencies", PROC, None, [("Textures", "proc2", dict(freqU=(0.25, 0.25, 0.25),
                                                                 colorU=[(1.0, 0.0, 0.0), (0.0, 1.0, 0.0), (0.0, 0.0, 1.0)]))]),
    ("proc_power0", PROC, None, [("Lights", "l1", dict(power=0.0))]),
    ("zaphod_scaling", ZAPHOD, None, [("Textures", "paper", dict(scaling=0.5))]),
    ("sky_many", f"{TSC}/sky.sdl", None, [("Lights", "sun", dict(pos=(100.0, 50.0, -30.0))), ("Nodes", "b2", dict(shader="shiny")),
                                          ("Shaders", "matte", dict(kind="Phong")), ("Textures", "chk", dict(size=3.0))]),
]


def base_text(path, spare):
    text = read(path).replace('"../../scenes/skybox"', '"%s/skybox"' % SC)
    return add_entity(text, "Shaders", spare) if spare else text


def host_scene(tmp_path, path, spare, name="base"):
    d = tmp_path / name
    d.mkdir()
    return load_text(str(d), path, base_text(path, spare))


@pytest.mark.parametrize("name,path,spare,edits", CASES, ids=[c[0] for c in CASES])
def test_edits_match_the_edited_scene_file(tmp_path, name, path, spare, edits):
    s = host_scene(tmp_path, path, spare)
    desc_arrays(s)   # the flat description exists before the edit: it is updated in place
    for e in edits:
        apply_edit(s, e)
    text = base_text(path, spare)
    for e in edits:
        text = edit_text(text, e)
    d = tmp_path / "ref"
    d.mkdir()
    ref = load_text(str(d), path, text)
    assert_same_desc(desc_arrays(s), desc_arrays(ref))
    # and the same when the description is first built after the edits
    s2 = host_scene(tmp_path, path, spare, "late")
    for e in edits:
        apply_edit(s2, e)
    assert_same_desc(desc_arrays(s2), desc_arrays(ref))


def test_indices_address_the_same_entities_as_names(tmp_path):
    by_name, by_index = host_scene(tmp_path, CHESS, HIGHLIGHT, "a"), host_scene(tmp_path, CHESS, HIGHLIGHT, "b")
    assert by_index.index("shaders", "highlight") == 3 and by_index.index("lights", "sun") == 0
    by_name.set_node_shader("e2", "highlight")
    by_name.set_shader("floor_shader", texture=None)
    by_name.set_texture("board", size=4.0)
    by_name.set_light("sun", power=10.0)
    by_index.set_node_shader(by_index.index("nodes", "e2"), 3)
    by_index.set_shader(0, texture=None)
    by_index.set_texture(0, size=4.0)
    by_index.set_light(0, power=10.0)
    assert_same_desc(desc_arrays(by_name), desc_arrays(by_index))


def test_an_edit_changes_only_its_entries(tmp_path):
    s = host_scene(tmp_path, CHESS, HIGHLIGHT)
    before = desc_arrays(s)
    s.set_node_shader("e2", "highlight")
    after = desc_arrays(s)
    for k in before:
        if k != "node_shader":
            assert before[k].tobytes() == after[k].tobytes(), k
    assert list(np.flatnonzero(before["node_shader"] != after["node_shader"])) == [s.index("nodes", "e2")]
    assert after["node_shader"][s.index("nodes", "e2")] == 3


def test_bad_edits_are_refused_and_change_nothing(tmp_path):
    s = host_scene(tmp_path, LECTURE5, None)
    before = desc_arrays(s)
    n = s.info()
    refused = [
        lambda: s.set_node_shader(n["nodes"], "ball_shader"),        # node index out of range
        lambda: s.set_node_shader(-1, "ball_shader"),
        lambda: s.set_node_shader("floor", "no_such_shader"),
        lambda: s.set_shader(n["shaders"], color=(1, 1, 1)),
        lambda: s.set_shader("ball_shader", kind="Blinn"),          # unknown kind
        lambda: s.set_shader("ball_shader", texture="no_such_texture"),
        lambda: s.set_shader("floor_shader", exponent=3.0),         # a Phong key on a Lambert
        lambda: s.set_shader("ball_shader", kind="Lambert", strength=0.5),
        lambda: s.set_texture(n["textures"], scaling=1.0),
        lambda: s.set_texture("bmp", size=3.0),                      # a Checker key on a bitmap
        lambda: s.set_texture("bmp", freqU=(1, 2, 3)),
        lambda: s.set_light(n["lights"], power=1.0),
    ]
    for k, f in enumerate(refused):
        with pytest.raises(c2.C2rtError) as e:
            f()
        assert e.value.status == -1, k
    for f in (lambda: s.set_shader("no_such_shader", color=(1, 1, 1)), lambda: s.set_light("no_such_light", power=1.0),
              lambda: s.set_node_shader("floor", 99)):
        with pytest.raises(KeyError):
            f()
    with pytest.raises(ValueError):
        s.set_light("light1", pos=(1.0, 2.0))
    assert_same_desc(desc_arrays(s), before)


def test_raw_calls_fail_cleanly_without_a_scene():
    one = np.zeros(1, np.uint32)
    i32, f32, f64 = np.zeros(3, np.int32), np.zeros(18, np.float32), np.zeros(6, np.float64)
    calls = [
        lambda: api.lib.c2rt_scene_set_node_shaders(None, 1, one.ctypes.data, i32.ctypes.data),
        lambda: api.lib.c2rt_scene_set_shaders(None, 1, one.ctypes.data, i32.ctypes.data, f32.ctypes.data, i32.ctypes.data,
                                               f64.ctypes.data, f32.ctypes.data),
        lambda: api.lib.c2rt_scene_set_textures(None, 1, one.ctypes.data, f32.ctypes.data, f64.ctypes.data),
        lambda: api.lib.c2rt_scene_set_lights(None, 1, one.ctypes.data, f64.ctypes.data, f32.ctypes.data, f32.ctypes.data),
    ]
    for f in calls:
        assert f() == -1 and b"scene is null" in api.lib.c2rt_last_error()
    with pytest.raises(c2.C2rtError, match="scene is null"):
        c2.scene_set_lights(None, [0], [0.0, 1.0, 0.0], [1.0, 1.0, 1.0], [1.0])
    with pytest.raises(ValueError):
        c2.scene_set_shaders(None, [0, 1], [0], [1.0] * 6, [-1, -1], [0.0, 0.0], [0.0, 0.0])


def test_bindings_follow_the_header():
    for name, n_args in (("c2rt_scene_set_node_shaders", 4), ("c2rt_scene_set_shaders", 8), ("c2rt_scene_set_textures", 5),
                         ("c2rt_scene_set_lights", 6)):
        assert name in api.C_ABI_SYMBOLS
        f = getattr(api.lib, name)
        assert f.argtypes[1] is C.c_size_t and len(f.argtypes) == n_args
