"""Partial frames after edits (c2rt_render_update, HostScene.render_update): every frame is np.array_equal, rgb and argb, to a
fresh c2rt_render of the same scene state, across chess moves, captures, promotions and highlights at a tiled and a ragged
size, shadow-only changes, nodes leaving and entering the view, other scene classes (MODE_BIG, the global-memory form, nested
CSG), every full-frame trigger, ARGB-only delivery, ray counts, a seeded fuzz of node moves and two device contexts."""
import ctypes as C
import os
import threading

import numpy as np
import pytest

import chess2rt_b200 as c2
from chess2rt_b200 import api
from sdl_edit import SC, TSC

pytestmark = pytest.mark.gpu

CHESS = os.path.join(SC, "chessboard.sdl")
LECTURE5 = os.path.join(SC, "lecture5.sdl")
PROC = os.path.join(SC, "lecture4-proc-texture.sdl")
ZAPHOD = os.path.join(SC, "zaphod.sdl")
NESTED = os.path.join(TSC, "nested.sdl")
STEREO = os.path.join(TSC, "stereo.sdl")


@pytest.fixture
def ctx():
    c2.init(1, [0])
    yield
    c2.init(1, [0])


def load(path, size):
    s = c2.HostScene(path)
    s.set_frame_size(*size)
    return s


def check(s, full=None, partial=False, argb_only=False, count_rays=False, seed=0):
    """One render_update, held bit for bit against render() of the same state; returns (info, update stats)."""
    ref_rgb, ref_argb, ref_st = s.render(argb=True, argb_only=argb_only, seed=seed, count_rays=count_rays)
    rgb, argb, st, info = s.render_update(argb=True, argb_only=argb_only, seed=seed, count_rays=count_rays)
    assert np.array_equal(argb, ref_argb), info
    if not argb_only:
        assert np.array_equal(rgb.view(np.uint32), ref_rgb.view(np.uint32)), info
    assert info["tiles_total"] == -(-s.frame_size[0] // 16) * -(-s.frame_size[1] // 8)
    if full is not None:
        assert info["full"] == full, info
    if info["full"]:
        assert info["tiles_rendered"] == info["tiles_total"]
        if count_rays:
            assert (st.primary_rays, st.shadow_rays) == (ref_st.primary_rays, ref_st.shadow_rays)
    if partial:
        assert not info["full"] and 0 < info["tiles_rendered"] < info["tiles_total"], info
    return info, st


def chess_sequence(s):
    """First frame, a no-op, pawn e2-e4 in four steps, a capture, a promotion, a highlight and its undo, the move back."""
    check(s, full=True)
    info, _ = check(s, full=False)
    assert info["tiles_rendered"] == 0
    for z in (-45.0, -40.0, -35.0, -30.0):
        s.place_node("e2", translate=(10.0, 0.0, z))
        check(s, partial=True)
    s.place_node("d7", translate=(130.0, 0.0, 40.0))
    check(s, partial=True)
    s.place_node("a7", geometry="queen", translate=(-70.0, 0.0, 70.0))
    check(s, partial=True)
    s.set_node_shader("e2", "black_piece")
    check(s, partial=True)
    s.set_node_shader("e2", "white_piece")
    check(s, partial=True)
    s.place_node("e2", translate=(10.0, 0.0, -50.0))
    check(s, partial=True)


@pytest.mark.parametrize("size", [(240, 135), (197, 111)])
def test_chess_moves_give_the_full_frame_bits(ctx, size):
    chess_sequence(load(CHESS, size))


def test_shadow_only_change(ctx):
    """A pawn above the top of the view (no camera ray can reach it) whose shadow falls on the board: moving it changes pixels,
    and only the shadow test can find them."""
    s = load(CHESS, (240, 135))
    s.place_node("h2", translate=(-55.0, 130.0, -55.0))
    check(s, full=True)
    before = s.render(argb_only=True)[1].copy()
    s.place_node("h2", translate=(-45.0, 130.0, -50.0))
    info, _ = check(s, partial=True)
    assert not np.array_equal(before, s.render(argb_only=True)[1])   # the shadow moved


def test_nodes_leave_and_enter_the_view(ctx):
    s = load(CHESS, (240, 135))
    check(s, full=True)
    s.place_node("b2", translate=(0.0, 0.0, -900.0))   # behind the camera
    check(s, partial=True)
    s.place_node("g7", translate=(900.0, 0.0, 0.0))    # far off to the side
    check(s, partial=True)
    s.place_node("b2", translate=(0.0, 0.0, 10.0))     # back onto the board
    check(s, partial=True)
    s.place_node("g7", translate=(-10.0, 0.0, 30.0))
    check(s, partial=True)


def test_lecture5_and_nested(ctx):
    s = load(LECTURE5, (320, 200))
    check(s, full=True)
    for t in ((100.0, 15.0, 240.0), (90.0, 25.0, 230.0), (100.0, 15.0, 256.0)):
        s.place_node(3, translate=t)
        check(s, full=False)
    n = load(NESTED, (160, 100))
    check(n, full=True)
    n.place_node("c", translate=(0.0, 30.0, 20.0))
    check(n, full=False)
    n.place_node("d", geometry="deeper", translate=(70.0, 20.0, -20.0))
    check(n, full=False)


def test_big_scene_and_global_records(ctx, tmp_path, monkeypatch):
    from test_gpu_parity import big_scene_text
    p = tmp_path / "big.sdl"
    p.write_text(big_scene_text(16))
    s = load(str(p), (200, 120))
    assert s.info()["nodes"] == 257
    check(s, full=True)
    for k, t in enumerate(((10.0, 6.0, 10.0), (-30.0, 8.0, 20.0), (0.0, 40.0, 0.0))):
        s.place_node("n%d" % (37 * k + 5), translate=t)
        check(s, full=False)
    monkeypatch.setenv("C2RT_FORCE_GLOBAL", "1")
    g = load(CHESS, (240, 135))
    check(g, full=True)   # the scene is created (and its class fixed) at its first frame
    monkeypatch.delenv("C2RT_FORCE_GLOBAL")
    g.place_node("e2", translate=(10.0, 0.0, -30.0))
    check(g, partial=True)
    g.set_node_shader("e2", "black_piece")
    check(g, partial=True)


MODE_SCENE = """Scene { GlobalSettings { frameWidth 160; frameHeight 96; ambientLightColor 0.1 0.1 0.1; AAEnabled true; prepassEnabled false }
 Camera { pos 0 30 -60; yaw 0; pitch -20; roll 0; fov 60 }
 Lights { PointLight "l" { pos -50 100 -40; color 1 1 1; power 30000 } }
 Geometries { Plane "floor" { y 0 }; Sphere "s" { center 0 0 0; R 5 } }
 Shaders { Lambert "f" { color 0.8 0.8 0.8 }; Lambert "a" { color 0.9 0.3 0.2 } }
 Nodes { Node "floor" { geometry "floor"; shader "f" }; Node "a" { geometry "s"; shader "a"; translate -8 5 0 };
         Node "b" { geometry "s"; shader "a"; translate 8 5 0 } } }
"""


def test_every_full_frame_trigger(ctx, tmp_path):
    s = load(CHESS, (240, 135))
    check(s, full=True)
    s.camera_move(1.0, 0.0, 0.0)
    check(s, full=True)                       # camera
    check(s, full=True, seed=3)               # settings
    check(s, full=False, seed=3)
    s.set_frame_size(200, 120)
    check(s, full=True)                       # frame size
    s.set_light("sun", power=70000.0)
    check(s, full=True)                       # light
    s.set_shader("white_piece", color=(0.9, 0.8, 0.7))
    check(s, full=True)                       # shader
    check(s, full=True, argb_only=True)       # other output buffers
    check(s, full=False, argb_only=True)
    p = tmp_path / "mode.sdl"
    p.write_text(MODE_SCENE)
    m = load(str(p), (160, 96))
    check(m, full=True)
    m.place_node("a", translate=(-6.0, 5.0, 0.0))
    check(m, partial=True)
    m.place_node("a", rotate=(0.0, 20.0, 0.0), translate=(-6.0, 5.0, 0.0))   # the scene becomes generic
    check(m, full=True)
    for path, size in ((ZAPHOD, (160, 100)), (STEREO, (160, 100)), (PROC, (160, 100))):   # DOF, stereo, one plane
        d = load(path, size)
        check(d, full=True)
        check(d, full=True)


def test_frame_after_a_cancel_is_full(ctx):
    """A c2rt_cancel that reaches an update frame in flight: C2RT_CANCELLED, and the next frame is a full one.  One attempt:
    when the cancel lands after the frame has finished it cancels nothing, and the test is skipped."""
    s = load(CHESS, (3840, 2160))
    check(s, full=True, argb_only=True)
    s.camera_move(0.0, 0.0, 0.5)   # a full frame, long enough for the cancel to land
    t = threading.Timer(0.001, api.lib.c2rt_cancel)
    t.start()
    s.render_update(argb_only=True)
    t.join()
    if not s.cancelled:
        pytest.skip("the cancel arrived after the frame")
    check(s, full=True, argb_only=True)
    check(s, full=False, argb_only=True)


def test_count_rays_and_argb_only(ctx):
    s = load(CHESS, (240, 135))
    check(s, full=True, argb_only=True, count_rays=True)
    _, st = check(s, full=False, argb_only=True, count_rays=True)
    assert (st.primary_rays, st.shadow_rays) == (0, 0)
    s.place_node("e2", translate=(10.0, 0.0, -40.0))
    info, st = check(s, partial=True, argb_only=True, count_rays=True)
    full = s.render(argb_only=True, count_rays=True)[2]
    # 5 AA taps per pixel of the rendered tiles (none of the chess frame's tiles is ragged at 240 x 135 but the last row)
    assert 0 < st.primary_rays <= 5 * 128 * info["tiles_rendered"] and st.primary_rays < full.primary_rays
    assert st.shadow_rays < full.shadow_rays


def test_fuzz_node_moves(ctx):
    from scene_fuzz import generate
    import tempfile
    rng = np.random.default_rng(14)
    with tempfile.TemporaryDirectory() as d:
        for seed in range(40):
            p = os.path.join(d, "f%d.sdl" % seed)
            with open(p, "w") as f:
                f.write(generate(seed))
            s = c2.HostScene(p)
            n = s.info()["nodes"]
            check(s, full=True)
            for _ in range(10):
                i = int(rng.integers(n))
                t = rng.normal(0.0, 8.0, 3)
                try:
                    s.place_node(i, translate=t)
                except c2.C2rtError:
                    continue
                check(s)
            s.close()


@pytest.mark.parametrize("devices", ["dev0x2", "distinct"])
def test_two_devices(devices):
    if devices == "distinct":
        if c2.device_count() < 2:
            pytest.skip("needs >= 2 GPUs")
        ids = [0, 1]
    else:
        ids = [0, 0]
    try:
        c2.init(2, ids)
        chess_sequence(load(CHESS, (240, 135)))
        chess_sequence(load(CHESS, (197, 111)))
        s = load(CHESS, (640, 360))   # several bands per device
        check(s, full=True)
        s.place_node("e2", translate=(10.0, 0.0, -30.0))
        check(s, partial=True)
    finally:
        c2.init(1, [0])
