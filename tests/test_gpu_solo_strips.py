"""Strips of the one-plane frame kernel (render_kernel.cu render_solo_kernel): a CTA renders several consecutive 32x8 tiles of
its tile row with one row table and one warp vote for the whole strip, and votes again per tile where the strip vote fails.
Every frame must be BIT-identical to the general kernel (C2RT_NO_SOLO_FAST=1), the ARGB plane and the ray counts included.
C2RT_SOLO_STRIP=n sets the strip width (test frames are small enough that the launch would otherwise keep one tile per CTA).
A numpy replay of the vote at strip level (test_gpu_solo_uniform.warp_paths with the tile width set to the strip width) must
find strips that pass and strips that fail while some of their tiles pass: the Procedure2 bound and a low light falling
inside a strip.  Widths where the last strip is short or narrower than a tile, heights that are not multiples of 8, row bands,
AA on and off, ARGB-only delivery and a rolled camera (no row table, one tile per CTA) cover the loop's edges."""
import os

import numpy as np
import pytest

import chess2rt_b200 as c2
import test_gpu_solo_uniform as uniform
from test_gpu_solo_rows import assert_same_as_general, level_scene
from test_gpu_solo_tiles import fast_and_general, render_device_bands

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SC = os.path.join(ROOT, "scenes")


@pytest.fixture(scope="module", autouse=True)
def _ctx():
    c2.init(1, [0])
    yield
    c2.shutdown()


def paths(g, name, width):
    """warp_paths with `width` columns per vote: 32 replays the per-tile vote, 32 s the strip vote."""
    saved = uniform.TILE_W
    uniform.TILE_W = width
    try:
        return uniform.warp_paths(g, name)
    finally:
        uniform.TILE_W = saved


def check_strip_frame(g, name, s, monkeypatch, what):
    """The replay first: strips that certainly pass, strips that certainly fail, and a failing strip with a tile that certainly
    passes.  With whole strips (s divides the tiles of a row) the failing strips cover s x (their number) warp tiles; when
    fewer warp tiles than that fail or are unsure, one of them passes.  Then the frame against the general kernel."""
    w, h = g.frame_size
    tiles_x = (w + 31) // 32
    assert tiles_x % s == 0, (w, s)
    t_pass, _, _ = paths(g, name, 32)
    s_pass, s_fail, why = paths(g, name, 32 * s)
    tiles = (h + uniform.WARP_ROWS - 1) // uniform.WARP_ROWS * tiles_x   # warp tiles: a warp's rows x 32 columns
    assert s_pass > 0 and s_fail > 0 and tiles - t_pass < s * s_fail, (what, s_pass, s_fail, why, t_pass, tiles)
    monkeypatch.setenv("C2RT_SOLO_STRIP", str(s))
    assert_same_as_general(g, monkeypatch, what)
    return why


@pytest.mark.parametrize("s", [2, 5])
@pytest.mark.parametrize("yaw", [0.0, 23.0, -61.0])
def test_procedure2_bound_inside_a_strip(yaw, s, monkeypatch):
    name = "../tests/scenes/proc_far.sdl"
    g = level_scene(name, {}, 2.0, -45.0)
    g.camera_rotate(yaw, 0.0, -45.0)
    g.set_frame_size(320, 187)
    why = check_strip_frame(g, name, s, monkeypatch, f"proc_far yaw {yaw} strips of {s}")
    assert why["sine range"] > 0, why


@pytest.mark.parametrize("s", [2, 5])
@pytest.mark.parametrize("yaw", [0.0, 15.0])
def test_low_light_inside_a_strip(yaw, s, monkeypatch):
    name = "../tests/scenes/proc_light_low.sdl"
    g = level_scene(name, {}, 0.0, -30.0)
    g.camera_rotate(yaw, 0.0, -30.0)
    g.set_frame_size(320, 240)
    why = check_strip_frame(g, name, s, monkeypatch, f"proc_light_low yaw {yaw} strips of {s}")
    assert why["near light"] > 0, why


# widths: a single column, one tile short and over, four tiles short and over, and strips that do not divide the row
WIDTHS = (1, 31, 33, 127, 129, 333)
HEIGHTS = (1, 9, 187)


@pytest.mark.parametrize("aa", [1, 0])
@pytest.mark.parametrize("s", [2, 3, 8])
@pytest.mark.parametrize("name,over,level", [("lecture4-proc-texture.sdl", {}, True), ("lecture4.sdl", {}, True),
                                             ("../tests/scenes/sky_plane.sdl", {}, False)])
def test_ragged_strips_equal_the_general_kernel(name, over, level, s, aa, monkeypatch):
    """sky_plane keeps its camera's roll: its kernel (no row table) keeps one tile per CTA whatever C2RT_SOLO_STRIP says."""
    g = level_scene(name, over, 0.0, -30.0) if level else c2.HostScene(os.path.join(SC, name))
    g.override(aa=aa, **over)
    if level:
        g.camera_rotate(17.0, 0.0, -20.0)
    monkeypatch.setenv("C2RT_SOLO_STRIP", str(s))
    lit = 0.0
    for w in WIDTHS:
        for h in HEIGHTS:
            g.set_frame_size(w, h)
            (rgb, argb, st), (rgb_g, argb_g, st_g) = fast_and_general(monkeypatch, lambda: g.render(argb=True, seed=5, count_rays=True))
            what = f"{name} aa={aa} strips of {s} {w}x{h}"
            np.testing.assert_array_equal(rgb, rgb_g, err_msg=what)
            np.testing.assert_array_equal(argb, argb_g, err_msg=what)
            assert (st.primary_rays, st.shadow_rays) == (st_g.primary_rays, st_g.shadow_rays), what
            assert st.primary_rays == w * h * (5 if aa else 1), what
            lit = max(lit, float(rgb.max()))
    assert lit > 0.05


@pytest.mark.parametrize("s", [2, 4])
@pytest.mark.parametrize("name", ["lecture4-proc-texture.sdl", "../tests/scenes/sky_plane.sdl"])
def test_argb_only_strips(name, s, monkeypatch):
    g = c2.HostScene(os.path.join(SC, name))
    g.override(aa=1)
    monkeypatch.setenv("C2RT_SOLO_STRIP", str(s))
    for w, h in ((333, 187), (66, 7), (3, 1)):
        g.set_frame_size(w, h)
        (none, only, _), (_, only_g, _) = fast_and_general(monkeypatch, lambda: g.render(argb_only=True, seed=5))
        _, both_a, _ = g.render(argb=True, seed=5)
        assert none is None
        np.testing.assert_array_equal(only, only_g)
        np.testing.assert_array_equal(only, both_a)


@pytest.mark.parametrize("compact", [0, 1])
@pytest.mark.parametrize("name", ["lecture4-proc-texture.sdl", "../tests/scenes/proc_light_low.sdl"])
def test_row_bands_with_strips(name, compact, monkeypatch):
    """3 ranks' bands on one GPU, reassembled: the strips of a CTA lie in its global tile row."""
    g = level_scene(name, {}, 0.0, -30.0)
    g.camera_rotate(9.0, 0.0, 6.0 if name == "lecture4-proc-texture.sdl" else -30.0)
    monkeypatch.setenv("C2RT_SOLO_STRIP", "3")
    for w in (333, 330):
        g.set_frame_size(w, 187)
        (rgb, argb), (rgb_g, argb_g) = fast_and_general(monkeypatch, lambda: render_device_bands(g, 3, 16, compact))
        np.testing.assert_array_equal(rgb, rgb_g)
        np.testing.assert_array_equal(argb, argb_g)
        full, full_a, _ = g.render(argb=True, seed=5)
        np.testing.assert_array_equal(rgb, full)
        np.testing.assert_array_equal(argb, full_a)
