"""Shading and light edits in place (c2rt_scene_set_node_shaders / _set_shaders / _set_textures / _set_lights, HostScene.set_*):
after an edit every call on the uploaded scene gives the bits of a scene created fresh from the edited scene file — colour
frames (RGB and ARGB), hit frames, the pixel pick, ray queries, visibility and shaded rays — across scene classes (MODE_SOLO's
shader / texture swap, MODE_UPAT, MODE_PHONG, solo_fast), the global-memory form, GI refusal, the device route, a frame on
another thread, and two devices."""
import ctypes as C
import threading
import time

import numpy as np
import pytest

import chess2rt_b200 as c2
from chess2rt_b200 import api
from sdl_edit import SC, TSC
from sdl_shading import (add_entity, apply_edit, assert_same, bits, differs, edit_entity, edit_text, load_text, ray_set,
                         read, scene_outputs)

SIZE = (160, 90)
CHESS = f"{SC}/chessboard.sdl"
LECTURE5 = f"{SC}/lecture5.sdl"
PROC = f"{SC}/lecture4-proc-texture.sdl"
ZAPHOD = f"{SC}/zaphod.sdl"
SKY = f"{TSC}/sky.sdl"
HIGHLIGHT = 'Phong "highlight" { color 0.25 0.875 0.25; exponent 20 }'
FILL = 'PointLight "fill" { pos 300 400 -100; color 0.5 0.5 0.75; power 300000 }'
# a one-plane scene whose node uses shader 1 and shader 1 texture 1: MODE_SOLO swaps both into record 0
SWAP_TEX = 'Checker "chk" { color1 0.125 0.25 0.5; color2 1 0.875 0.75; size 17 }'
SWAP_SHADER = 'Phong "s1" { color 0.75 0.75 0.5; texture "chk"; exponent 12; strength 0.5 }'


@pytest.fixture(scope="module")
def ctx():
    c2.init(1, [0])
    yield
    c2.shutdown()


def base_text(path, extra=()):
    text = read(path).replace('"../../scenes/skybox"', '"%s/skybox"' % SC)
    for section, block in extra:
        text = add_entity(text, section, block)
    return text


def swap_text():
    text = base_text(PROC, [("Textures", SWAP_TEX), ("Shaders", SWAP_SHADER)])
    return edit_entity(text, "Nodes", "floor", shader="s1")


class Run:
    """A scene uploaded once and edited step by step, against a scene created fresh from the edited text after every step."""

    def __init__(self, tmp_path, path, text, size=SIZE):
        self.tmp, self.path, self.text, self.size, self.n = tmp_path, path, text, size, 0
        self.scene = self.fresh()
        self.rays = ray_set(self.scene)
        self.orig = scene_outputs(self.scene, self.rays)   # uploaded and resident before the first edit

    def fresh(self):
        self.n += 1
        d = self.tmp / ("s%d" % self.n)
        d.mkdir()
        return load_text(str(d), self.path, self.text, self.size)

    def step(self, *edits, what=""):
        before = scene_outputs(self.scene, self.rays)
        for e in edits:
            apply_edit(self.scene, e)
            self.text = edit_text(self.text, e)
        after = scene_outputs(self.scene, self.rays)
        assert_same(after, scene_outputs(self.fresh(), self.rays), what)
        assert differs(before, after), ("the edit changed nothing", what)
        return after


# (id, scene, scene text, [steps]); each step is a list of edits (section, entity, keys), checked against a fresh scene
CASES = [
    ("chess_highlight_and_back", CHESS, lambda: base_text(CHESS, [("Shaders", HIGHLIGHT)]),
     [[("Nodes", "e2", dict(shader="highlight"))], [("Nodes", "e2", dict(shader="white_piece"))]]),
    ("chess_checker", CHESS, lambda: base_text(CHESS),
     [[("Textures", "board", dict(color1=(0.5, 0.125, 0.0), color2=(1.0, 1.0, 0.75)))], [("Textures", "board", dict(size=12.5))]]),
    ("chess_piece_theme", CHESS, lambda: base_text(CHESS),
     [[("Shaders", "white_piece", dict(color=(0.875, 0.5, 0.25), exponent=8.0, strength=0.25))],
      [("Shaders", "black_piece", dict(kind="Lambert", color=(0.25, 0.125, 0.5)))]]),
    ("lecture5_relight", LECTURE5, lambda: base_text(LECTURE5),
     [[("Lights", "light1", dict(pos=(-200.0, 500.0, 100.0), color=(1.0, 0.75, 0.5), power=6e5))]]),
    ("lecture5_bitmap_switch", LECTURE5, lambda: base_text(LECTURE5),
     [[("Shaders", "csg_shader", dict(texture="world"))], [("Shaders", "floor_shader", dict(texture="world"))]]),
    ("proc_upat", PROC, lambda: base_text(PROC),
     [[("Textures", "proc2", dict(freqU=(0.25, 0.25, 0.25)))], [("Textures", "proc2", dict(freqU=(0.01, 0.25, 0.01)))]]),
    ("proc_phong_and_back", PROC, lambda: base_text(PROC),
     [[("Shaders", "floor_shader", dict(kind="Phong", texture="proc2", exponent=10.0))],
      [("Shaders", "floor_shader", dict(kind="Lambert", texture="proc2"))]]),
    ("proc_light_other_side_and_back", PROC, lambda: base_text(PROC),
     [[("Lights", "l1", dict(pos=(-30.0, -100.0, 250.0)))], [("Lights", "l1", dict(pos=(-30.0, 100.0, 250.0)))]]),
    ("proc_power0_and_back", PROC, lambda: base_text(PROC),
     [[("Lights", "l1", dict(power=0.0))], [("Lights", "l1", dict(power=50000.0))]]),
    ("solo_swap_by_description_index", PROC, swap_text,
     [[("Textures", "chk", dict(color1=(0.5, 0.0, 0.25), size=9.0)), ("Shaders", "floor_shader", dict(color=(0.5, 0.5, 0.5)))],
      [("Shaders", "s1", dict(color=(0.25, 0.5, 1.0), exponent=30.0))],
      [("place", "floor", dict(scale=(-1.0, 1.0, 1.0)))],                           # leaves MODE_SOLO (a mirrored plane)
      [("Shaders", "s1", dict(strength=0.875)), ("Textures", "proc2", dict(freqV=(0.5, 0.5, 0.125)))],
      [("Nodes", "floor", dict(shader="floor_shader"))],
      [("place", "floor", dict())],                                                 # back in MODE_SOLO, now on shader 0
      [("Textures", "proc2", dict(freqU=(0.125, 0.125, 0.125))), ("Nodes", "floor", dict(shader="s1"))],
      [("Textures", "chk", dict(size=4.0))]]),
    ("zaphod_dof_scaling", ZAPHOD, lambda: base_text(ZAPHOD), [[("Textures", "paper", dict(scaling=0.5))]]),
    ("two_lights_one_dimmed", LECTURE5, lambda: base_text(LECTURE5, [("Lights", FILL)]),
     [[("Lights", "fill", dict(power=0.0))], [("Lights", "light1", dict(color=(0.5, 1.0, 0.5)))]]),
    ("cubemap", SKY, lambda: base_text(SKY),
     [[("Lights", "sun", dict(pos=(100.0, 150.0, -30.0)))], [("Nodes", "b2", dict(shader="shiny")), ("Shaders", "matte", dict(kind="Phong"))],
      [("Textures", "chk", dict(size=3.0))]]),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,path,text,steps", CASES, ids=[c[0] for c in CASES])
def test_edits_give_the_fresh_scene_bits(ctx, tmp_path, name, path, text, steps):
    r = Run(tmp_path, path, text())
    for k, edits in enumerate(steps):
        r.step(*edits, what=(name, k))


@pytest.mark.gpu
def test_highlight_then_unhighlight_gives_the_original_bits(ctx, tmp_path):
    r = Run(tmp_path, CHESS, base_text(CHESS, [("Shaders", HIGHLIGHT)]))
    r.step(("Nodes", "e2", dict(shader="highlight")), ("Nodes", "d1", dict(shader="highlight")))
    r.step(("Nodes", "e2", dict(shader="white_piece")), ("Nodes", "d1", dict(shader="white_piece")))
    assert_same(scene_outputs(r.scene, r.rays), r.orig)


@pytest.mark.gpu
def test_global_memory_form(ctx, tmp_path, monkeypatch):
    monkeypatch.setenv("C2RT_FORCE_GLOBAL", "1")   # read at scene-create time, by both scenes
    r = Run(tmp_path, CHESS, base_text(CHESS, [("Shaders", HIGHLIGHT)]))
    r.step(("Nodes", "e2", dict(shader="highlight")), ("Lights", "sun", dict(pos=(50.0, 200.0, -100.0))))
    r.step(("Textures", "board", dict(size=5.0)), ("Shaders", "white_piece", dict(kind="Lambert")))


@pytest.mark.gpu
def test_gi_refusal_follows_the_edited_shaders(ctx, tmp_path):
    """A GI frame refuses Phong-shaded nodes: switching every Phong node's shader to Lambert makes it render (and equal a fresh
    scene's), switching one back makes it refuse again."""
    r = Run(tmp_path, CHESS, base_text(CHESS))
    s = r.scene

    def gi_frame(scene):
        cam, st = scene.frame_blocks(seed=3)
        st.gi_enabled, st.paths_per_pixel = 1, 2
        rgb = np.empty((st.frame_height, st.frame_width, 3), np.float32)
        rc = api.lib.c2rt_render(scene.device_scene(), C.byref(cam), C.byref(st), rgb.ctypes.data, None, None)
        return rc, bits(rgb) if rc == 0 else api.lib.c2rt_last_error()

    assert gi_frame(s)[0] < 0
    r.step(("Shaders", "white_piece", dict(kind="Lambert")), ("Shaders", "black_piece", dict(kind="Lambert")))
    rc, img = gi_frame(s)
    assert rc == 0, img
    rc_f, img_f = gi_frame(r.fresh())
    assert rc_f == 0 and np.array_equal(img, img_f)
    r.step(("Shaders", "black_piece", dict(kind="Phong")))
    rc, msg = gi_frame(s)
    assert rc < 0 and b"Phong" in msg, msg


@pytest.mark.gpu
def test_refused_edits_change_no_output(ctx):
    s = c2.HostScene(PROC)
    s.set_frame_size(*SIZE)
    rays = ray_set(s)
    orig = scene_outputs(s, rays)
    h = s.device_scene()
    i = np.zeros(1, np.uint32)
    bad = [
        lambda: c2.scene_set_node_shaders(h, [1], [0]),                                   # node out of range
        lambda: c2.scene_set_node_shaders(h, [0], [1]),                                   # shader out of range
        lambda: c2.scene_set_node_shaders(h, [0, 0], [0, -1]),                            # ... after a valid entry
        lambda: c2.scene_set_shaders(h, [1], [0], [1, 1, 1], [-1], [1.0], [1.0]),         # shader out of range
        lambda: c2.scene_set_shaders(h, [0], [7], [1, 1, 1], [-1], [1.0], [1.0]),         # unknown type
        lambda: c2.scene_set_shaders(h, [0], [1], [1, 1, 1], [1], [1.0], [1.0]),          # texture out of range
        lambda: c2.scene_set_textures(h, [1], np.zeros(18), np.ones(6)),                 # texture out of range
        lambda: c2.scene_set_lights(h, [0, 1], np.zeros(6), np.ones(6), [1.0, 1.0]),    # light out of range
        lambda: s.set_node_shader("floor", "no_such_shader"),
        lambda: s.set_shader("floor_shader", exponent=2.0),
        lambda: s.set_texture("proc2", scaling=2.0),
    ]
    for k, f in enumerate(bad):
        with pytest.raises(c2.C2rtError) as e:
            f()
        assert e.value.status == -1, k
    for f in (lambda: api.lib.c2rt_scene_set_node_shaders(h, 1, i.ctypes.data, None),
              lambda: api.lib.c2rt_scene_set_textures(h, 1, None, None, None),
              lambda: api.lib.c2rt_scene_set_lights(h, 1, i.ctypes.data, None, None, None)):
        assert f() == -1
    for f in (api.lib.c2rt_scene_set_node_shaders, api.lib.c2rt_scene_set_textures):   # n == 0: a no-op
        assert f(h, 0, *([None] * (len(f.argtypes) - 2))) == 0
    assert_same(scene_outputs(s, rays), orig)


@pytest.mark.gpu
def test_raw_edits_by_description_index_and_later_entries_win(ctx, tmp_path):
    """The raw calls address the description's indices, also when MODE_SOLO has swapped shader 1 / texture 1 into record 0."""
    r = Run(tmp_path, PROC, swap_text())
    h = r.scene.device_scene()
    d = r.scene.desc().contents
    colors = np.array([d.tex_colors[18 + k] for k in range(18)], np.float32)
    params = np.array([d.tex_params[6 + k] for k in range(6)])
    params[0] = 5.0
    c2.scene_set_textures(h, [1, 1], np.stack([colors, colors]), np.stack([np.ones(6), params]))
    c2.scene_set_shaders(h, [1], [1], [0.5, 0.25, 1.0], [1], [12.0], [0.5])
    c2.scene_set_lights(h, [0], [-30.0, 100.0, 250.0], [1.0, 0.5, 0.5], [40000.0])
    r.text = edit_text(r.text, ("Textures", "chk", dict(size=5.0)))
    r.text = edit_text(r.text, ("Shaders", "s1", dict(color=(0.5, 0.25, 1.0))))
    r.text = edit_text(r.text, ("Lights", "l1", dict(color=(1.0, 0.5, 0.5), power=40000.0)))
    assert_same(scene_outputs(r.scene, r.rays), scene_outputs(r.fresh(), r.rays))


@pytest.mark.gpu
def test_edit_while_another_scene_is_resident(ctx, tmp_path):
    a = Run(tmp_path, CHESS, base_text(CHESS, [("Shaders", HIGHLIGHT)]))
    b = c2.HostScene(LECTURE5)
    b.set_frame_size(*SIZE)
    rays_b = ray_set(b)
    b_before = scene_outputs(b, rays_b)   # b is now the resident scene
    apply_edit(a.scene, ("Nodes", "e2", dict(shader="highlight")))
    a.text = edit_text(a.text, ("Nodes", "e2", dict(shader="highlight")))
    assert_same(scene_outputs(b, rays_b), b_before)
    assert_same(scene_outputs(a.scene, a.rays), scene_outputs(a.fresh(), a.rays))


@pytest.mark.gpu
def test_device_route_after_an_edit_matches_the_host_route(ctx):
    import torch
    for path, edit in ((CHESS, ("Lights", "sun", dict(pos=(100.0, 250.0, -50.0)))), (PROC, ("Lights", "l1", dict(pos=(0.0, -50.0, 0.0))))):
        s = c2.HostScene(path)
        s.set_frame_size(192, 108)
        h = s.device_scene()
        stream = torch.cuda.Stream()
        w, hh = s.frame_size
        d_rgb = torch.empty(hh * w * 3, dtype=torch.float32, device="cuda")
        d_argb = torch.empty(hh * w, dtype=torch.int32, device="cuda")
        cam, st = s.frame_blocks(seed=1)
        api.render_device(h, cam, st, d_rgb.data_ptr(), d_argb.data_ptr(), stream=stream.cuda_stream)   # resident on the stream
        stream.synchronize()
        before = d_argb.cpu().numpy().copy()
        apply_edit(s, edit)
        cam, st = s.frame_blocks(seed=1)
        api.render_device(h, cam, st, d_rgb.data_ptr(), d_argb.data_ptr(), stream=stream.cuda_stream)
        stream.synchronize()
        rgb, argb, _ = s.render(argb=True, seed=1)
        assert np.array_equal(bits(d_rgb.cpu().numpy()), bits(rgb.reshape(-1))), path
        assert np.array_equal(d_argb.cpu().numpy().view(np.uint32), argb.reshape(-1)), path
        assert not np.array_equal(before, d_argb.cpu().numpy()), path


@pytest.mark.gpu
def test_an_edit_waits_for_a_frame_on_another_thread(ctx, tmp_path):
    """The edit takes the library lock: a frame running on another thread completes as the pre-edit or the post-edit frame,
    never a mixture."""
    size = (1920, 1080)
    r = Run(tmp_path, CHESS, base_text(CHESS, [("Shaders", HIGHLIGHT)]), size=(16, 16))
    s = r.scene
    s.set_frame_size(*size)
    cam, st = s.frame_blocks(seed=2)
    h = s.device_scene()

    def frame():
        rgb = np.empty((size[1], size[0], 3), np.float32)
        assert api.lib.c2rt_render(h, C.byref(cam), C.byref(st), rgb.ctypes.data, None, None) == 0
        return bits(rgb)

    pre = frame()
    frames, started = [], threading.Event()

    def worker():
        started.set()
        for _ in range(12):
            frames.append(frame())

    t = threading.Thread(target=worker)
    t.start()
    started.wait()
    time.sleep(0.002)
    # one call with two entries: a frame sees both or neither
    nodes = [s.index("nodes", "e2"), s.index("nodes", "d1")]
    c2.scene_set_node_shaders(h, nodes, [s.index("shaders", "highlight")] * 2)
    for node in ("e2", "d1"):
        r.text = edit_text(r.text, ("Nodes", node, dict(shader="highlight")))
    t.join()
    assert len(frames) == 12
    post_scene = r.fresh()
    post_scene.set_frame_size(*size)
    post_rgb, _, _ = post_scene.render(seed=2)
    post = bits(post_rgb)
    assert not np.array_equal(pre, post)
    for k, f in enumerate(frames):
        assert np.array_equal(f, pre) or np.array_equal(f, post), k
    assert np.array_equal(frame(), post)


@pytest.mark.gpu
@pytest.mark.skipif(c2.device_count() < 2, reason="needs two GPUs")
def test_two_devices_give_the_fresh_scene_bits(tmp_path):
    c2.init(2, [0, 1])
    try:
        r = Run(tmp_path, CHESS, base_text(CHESS, [("Shaders", HIGHLIGHT)]), size=(320, 180))
        r.step(("Nodes", "e2", dict(shader="highlight")), ("Lights", "sun", dict(pos=(50.0, 200.0, -100.0))),
               ("Textures", "board", dict(size=10.0)))
    finally:
        c2.init(1, [0])
