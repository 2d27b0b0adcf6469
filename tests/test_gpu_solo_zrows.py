"""The z half of the one-plane kernel's row table (render_kernel.cu render_solo_kernel<..., ROWS_YZ>, row_z): with no camera yaw
and no roll, du.z == 0 as well as du.y == 0, so a camera ray's d.z, its hit point's z, the texture's v part and the light
vector's z component are constants of the (row, AA tap), and the straight-line tap takes them from the table.  Every frame must
be BIT-identical to the general kernel (C2RT_NO_SOLO_FAST=1), the ARGB plane and the ray counts included.  Each case checks
from the camera block which kernel the frame takes: du.z == 0 (the z table) or != 0 (the rows kernel without it)."""
import os
import shutil

import numpy as np
import pytest

import chess2rt_b200 as c2
from test_gpu_solo_rows import assert_same_as_general, camera_rows
from test_gpu_solo_tiles import fast_and_general, render_device_bands

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SC = os.path.join(ROOT, "scenes")

TEXTURES = {
    "none": "",
    "checker": 'Checker "t" { color1 0.1 0.2 0.1; color2 0.9 0.8 0.3; size 7 }',
    "procedure2": """Procedure2 "t" {
      freqU 0.01 0.25 0.01
      freqV 0.01 0.25 0.01
      colorU { color 0.7 0.1 0.2; color 0.3 0.4 0.9; color 0.5 0.8 0.1 }
      colorV { color 0.5 0.8 0.1; color 0.7 0.1 0.2; color 0.3 0.4 0.9 }
    }""",
    "bitmap": 'BitmapTexture "t" { file "texture/zaphod.bmp"; assumedGamma 2.2 }',
}
SHADERS = {
    "lambert": 'Lambert "s" {{ color 0.9 0.8 0.7{tex} }}',
    "phong": 'Phong "s" {{ color 0.9 0.8 0.7; exponent 40; strength 1{tex} }}',
    "phong_sharp": 'Phong "s" {{ color 0.9 0.8 0.7; exponent 5000; strength 2{tex} }}',   # the FP64 lobe (exponent > 2048)
}


@pytest.fixture(scope="module", autouse=True)
def _ctx():
    c2.init(1, [0])
    yield
    c2.shutdown()


def write_scene(tmp_path, texture, shader):
    os.makedirs(tmp_path / "texture", exist_ok=True)
    shutil.copy(os.path.join(SC, "texture", "zaphod.bmp"), tmp_path / "texture" / "zaphod.bmp")
    tex = TEXTURES[texture]
    sh = SHADERS[shader].format(tex='; texture "t"' if tex else "")
    text = f"""Scene {{
  Name "zrows"
  GlobalSettings {{ frameWidth 320; frameHeight 187; ambientLightColor 0.05 0.05 0.05; AAEnabled true; prepassEnabled false }}
  Camera {{ pos 0 40 -100; yaw 0; pitch -30; roll 0; fov 90 }}
  Lights {{ PointLight "l" {{ pos 10 60 40; color 1 1 1; power 4000 }} }}
  Geometries {{ Plane "floor" {{ y 0 }} }}
  {"Textures { " + tex + " }" if tex else ""}
  Shaders {{ {sh} }}
  Nodes {{ Node "n" {{ geometry "floor"; shader "s" }} }}
}}
"""
    path = tmp_path / f"{texture}_{shader}.sdl"
    path.write_text(text)
    return c2.HostScene(str(path))


def du(g):
    cam, _ = g.frame_blocks(seed=5)
    return [cam.up_right[k] - cam.up_left[k] for k in range(3)]


def assert_z_table(g, expect=True):
    d = du(g)
    assert d[1] == 0.0, "a roll-free camera: the frame takes a row table"
    assert (d[2] == 0.0) == expect, ("du.z", d[2])


@pytest.mark.parametrize("shader", list(SHADERS))
@pytest.mark.parametrize("texture", list(TEXTURES))
def test_texture_and_shader_kinds_equal_the_general_kernel(texture, shader, tmp_path, monkeypatch):
    """Pitches with the horizon inside the frame, the camera looking down and up, ragged sizes."""
    g = write_scene(tmp_path, texture, shader)
    horizon, lit = 0, 0.0
    for d_pitch in (0.0, 24.0, 30.0, 10.0, -20.0):
        g.camera_rotate(0.0, 0.0, d_pitch)
        for w, h in ((320, 187), (333, 61), (66, 9)):
            g.set_frame_size(w, h)
            assert_z_table(g)
            dy, _ = camera_rows(g)
            below = np.signbit(dy).all(axis=1)
            horizon += bool(below.any() and not below.all())
            rgb = assert_same_as_general(g, monkeypatch, f"{texture} {shader} pitch {d_pitch} {w}x{h}")
            lit = max(lit, float(rgb.max()))
        g.camera_rotate(0.0, 0.0, -d_pitch)
    assert horizon > 0 and lit > 0.05, (horizon, lit)


@pytest.mark.parametrize("name", ["../tests/scenes/proc_far.sdl", "../tests/scenes/proc_light_low.sdl", "lecture4-proc-texture.sdl",
                                  "lecture4.sdl"])
def test_yaw_free_scenes_equal_the_general_kernel(name, monkeypatch):
    """proc_far: the Procedure2 bound inside tile rows (some warps on the per-ray loop); proc_light_low: pixels under a low light;
    forced strips as well as the launch's own."""
    g = c2.HostScene(os.path.join(SC, name))
    g.override(aa=1)
    if name == "../tests/scenes/proc_far.sdl":   # the file has yaw 12 and roll 2
        g.camera_rotate(-12.0, -2.0, 0.0)
    for s in (None, 2, 5):
        if s is None:
            monkeypatch.delenv("C2RT_SOLO_STRIP", raising=False)
        else:
            monkeypatch.setenv("C2RT_SOLO_STRIP", str(s))
        for w, h in ((320, 187), (330, 240)):
            g.set_frame_size(w, h)
            assert_z_table(g)
            assert_same_as_general(g, monkeypatch, f"{name} strips {s} {w}x{h}")


@pytest.mark.parametrize("aa", [1, 0])
def test_ragged_sizes_equal_the_general_kernel(aa, monkeypatch):
    g = c2.HostScene(os.path.join(SC, "lecture4-proc-texture.sdl"))
    g.override(aa=aa)
    monkeypatch.setenv("C2RT_SOLO_STRIP", "3")
    for w in (1, 31, 33, 129, 333):
        for h in (1, 9, 187):
            g.set_frame_size(w, h)
            assert_z_table(g)
            (rgb, argb, st), (rgb_g, argb_g, st_g) = fast_and_general(monkeypatch, lambda: g.render(argb=True, seed=5, count_rays=True))
            what = f"aa={aa} {w}x{h}"
            np.testing.assert_array_equal(rgb, rgb_g, err_msg=what)
            np.testing.assert_array_equal(argb, argb_g, err_msg=what)
            assert (st.primary_rays, st.shadow_rays) == (st_g.primary_rays, st_g.shadow_rays), what
            assert st.primary_rays == w * h * (5 if aa else 1), what


def test_argb_only_delivery(monkeypatch):
    g = c2.HostScene(os.path.join(SC, "lecture4-proc-texture.sdl"))
    for w, h in ((333, 187), (66, 7)):
        g.set_frame_size(w, h)
        assert_z_table(g)
        (none, only, _), (_, only_g, _) = fast_and_general(monkeypatch, lambda: g.render(argb_only=True, seed=5))
        _, both_a, _ = g.render(argb=True, seed=5)
        assert none is None
        np.testing.assert_array_equal(only, only_g)
        np.testing.assert_array_equal(only, both_a)


@pytest.mark.parametrize("compact", [0, 1])
def test_row_bands(compact, monkeypatch):
    """3 ranks' bands on one GPU, reassembled: the z table is built for the CTA's global rows."""
    g = c2.HostScene(os.path.join(SC, "lecture4-proc-texture.sdl"))
    for w in (333, 330):
        g.set_frame_size(w, 187)
        assert_z_table(g)
        (rgb, argb), (rgb_g, argb_g) = fast_and_general(monkeypatch, lambda: render_device_bands(g, 3, 16, compact))
        np.testing.assert_array_equal(rgb, rgb_g)
        np.testing.assert_array_equal(argb, argb_g)
        full, full_a, _ = g.render(argb=True, seed=5)
        np.testing.assert_array_equal(rgb, full)
        np.testing.assert_array_equal(argb, full_a)


@pytest.mark.parametrize("name", ["lecture4-proc-texture.sdl", "lecture4.sdl"])
def test_tiny_yaw_takes_the_rows_kernel(name, monkeypatch):
    """A yaw of 1e-9 degrees: du.z != 0, the frame runs on the rows kernel without the z table, and still matches."""
    g = c2.HostScene(os.path.join(SC, name))
    g.override(aa=1)
    g.camera_rotate(1e-9, 0.0, 0.0)
    g.set_frame_size(333, 187)
    assert_z_table(g, expect=False)
    assert_same_as_general(g, monkeypatch, f"{name} yaw 1e-9")
