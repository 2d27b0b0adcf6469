"""The per-row table of the one-plane frame kernel (render_kernel.cu render_solo_kernel<..., ROWS = true>, row_tap): with no
camera roll, du.y == 0 and a camera ray's d.y depends on its row and AA tap only, so the plane's sign test, grazing prefilter,
hit distance and the shadow ray's D.y are computed once per (row, tap).  Every frame must be BIT-identical to the general
kernel of the same scene class (C2RT_NO_SOLO_FAST=1, read per frame), the ARGB plane and the ray counts included: roll-free
cameras at several yaws and pitches, the horizon inside the frame, rays within a few ulps of horizontal (sign-test misses and
the per-ray grazing test), a camera below the plane, a rolled camera (per-ray path) and row bands."""
import os
from fractions import Fraction

import numpy as np
import pytest

import chess2rt_b200 as c2
from test_gpu_solo_tiles import fast_and_general, render_device_bands

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SC = os.path.join(ROOT, "scenes")

# (scene, overrides, camera roll and pitch in the file): procedural texture, checker, cubemap environment (misses go through
# env_lookup), bitmap, and an untextured Phong lobe of exponent 5000 (the FP64 lobe)
SCENES = [("lecture4-proc-texture.sdl", {}, 0.0, -30.0), ("lecture4.sdl", {}, 0.0, -30.0),
          ("../tests/scenes/sky_plane.sdl", {}, 5.0, 8.0), ("zaphod.sdl", {"dof": 0}, 2.3, -41.8),
          ("../tests/scenes/phong_sharp.sdl", {}, 0.0, -30.0)]
SIZES = ((333, 187), (130, 61), (66, 9))
KX, KY = (0.0, 0.3, 0.6, 0.0, 0.6), (0.0, 0.3, 0.0, 0.6, 0.6)   # AA tap offsets (renderer.d:235-242)


@pytest.fixture(scope="module", autouse=True)
def _ctx():
    c2.init(1, [0])
    yield
    c2.shutdown()


def level_scene(name, over, roll, pitch):
    """The scene with its camera's roll taken out and its pitch set to 0 (x + -x is exactly 0)."""
    g = c2.HostScene(os.path.join(SC, name))
    g.override(aa=1, **over)
    g.camera_rotate(0.0, -roll, -pitch)
    return g


def fma(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))   # exact product and sum, one rounding


def camera_rows(g):
    """d.y of every (row, AA tap) as render_kernel.cu screen_dir + tap_d form it, and c2rt_api.cu fill_params' grazing bound."""
    cam, st = g.frame_blocks(seed=5)
    assert cam.up_left[1] == cam.up_right[1], "a roll-free camera: du.y == 0, the frame takes the per-row table"
    inv_w, inv_h = 1.0 / cam.frame_width, 1.0 / cam.frame_height
    ul = [cam.up_left[k] - cam.pos[k] for k in range(3)]
    du = [cam.up_right[k] - cam.up_left[k] for k in range(3)]
    dv = [cam.down_left[k] - cam.up_left[k] for k in range(3)]
    tap = [du[1] * (KX[t] * inv_w) + dv[1] * (KY[t] * inv_h) for t in range(5)]
    inner = fma(du[1], 0.0 * inv_w, ul[1])
    dy = np.array([[fma(dv[1], y * inv_h, inner) + tap[t] for t in range(5)] for y in range(st.frame_height)])
    dmax2 = 0.0
    for c in range(4):
        sx = (st.frame_width + 2.0) * inv_w if c & 1 else -inv_w
        sy = (st.frame_height + 2.0) * inv_h if c & 2 else -inv_h
        l2 = 0.0
        for k in range(3):
            v = ul[k] + du[k] * sx + dv[k] * sy
            l2 += v * v
        dmax2 = max(dmax2, l2)
    return dy, 1e-18 * dmax2 * (1.0 + 1e-6)


def assert_same_as_general(g, monkeypatch, what):
    (rgb, argb, st), (rgb_g, argb_g, st_g) = fast_and_general(monkeypatch, lambda: g.render(argb=True, seed=5, count_rays=True))
    np.testing.assert_array_equal(rgb, rgb_g, err_msg=what)
    np.testing.assert_array_equal(argb, argb_g, err_msg=what)
    assert (st.primary_rays, st.shadow_rays) == (st_g.primary_rays, st_g.shadow_rays), what
    w, h = g.frame_size
    assert st.primary_rays == w * h * 5, what
    return rgb


@pytest.mark.parametrize("name,over,roll,pitch", SCENES)
def test_roll_free_cameras_equal_the_general_kernel(name, over, roll, pitch, monkeypatch):
    g = level_scene(name, over, roll, pitch)
    g.camera_rotate(0.0, 0.0, pitch)   # the file's view without its roll
    horizon, lit = 0, 0.0
    for d_yaw, d_pitch in ((0, 0), (17, -9), (-140, 25), (63, 12), (0, 4 - pitch), (25, -4 - pitch)):
        g.camera_rotate(d_yaw, 0.0, d_pitch)
        for w, h in SIZES:
            g.set_frame_size(w, h)
            dy, _ = camera_rows(g)
            below = np.signbit(dy).all(axis=1)   # rows whose rays all point down (the camera is above the plane here)
            horizon += bool(below.any() and not below.all())
            rgb = assert_same_as_general(g, monkeypatch, f"{name} yaw {d_yaw} pitch {d_pitch} {w}x{h}")
            lit = max(lit, float(rgb.max()))
        g.camera_rotate(-d_yaw, 0.0, -d_pitch)
    assert horizon > 0, "some frames have the horizon inside them"
    assert lit > 0.05


@pytest.mark.parametrize("name,over,roll,pitch", SCENES)
def test_near_horizontal_rays_equal_the_general_kernel(name, over, roll, pitch, monkeypatch):
    """Pitch 0 and pitches a few 1e-8 degrees off it, at even heights: the middle row's corner taps have d.y of +-0 or a few ulps
    (sign-test misses), or fall under the grazing prefilter, where grazing_exact decides per ray."""
    g = level_scene(name, over, roll, pitch)
    sign_miss = graze = 0
    for d_pitch in (0.0, 2e-9, -2e-9, 1e-8, -1e-8, 3e-8, -3e-8, 5e-8, -5e-8, 7e-8, -7e-8, 9e-8, -9e-8, 1.2e-7, -1.2e-7):
        g.camera_rotate(0.0, 0.0, d_pitch)
        for w, h in ((320, 180), (130, 62)):
            g.set_frame_size(w, h)
            dy, graze_dy2 = camera_rows(g)
            near = dy * dy < graze_dy2
            sign_miss += int((near & ~np.signbit(dy)).sum())   # above the plane: d.y = +0 or a few ulps up misses by the sign test
            graze += int((near & np.signbit(dy)).sum())
            assert_same_as_general(g, monkeypatch, f"{name} pitch {d_pitch} {w}x{h}")
        g.camera_rotate(0.0, 0.0, -d_pitch)
    assert sign_miss > 0 and graze > 0, (sign_miss, graze)


def test_camera_below_the_plane_equals_the_general_kernel(monkeypatch):
    g = c2.HostScene(os.path.join(ROOT, "tests", "scenes", "proc_below.sdl"))
    for d_yaw, d_pitch in ((0, 0), (50, 10), (-120, -20)):
        g.camera_rotate(d_yaw, 0.0, d_pitch)
        for w, h in SIZES:
            g.set_frame_size(w, h)
            dy, _ = camera_rows(g)
            assert (~np.signbit(dy)).any()   # the rays that reach the ceiling
            assert_same_as_general(g, monkeypatch, f"proc_below yaw {d_yaw} pitch {d_pitch} {w}x{h}")
        g.camera_rotate(-d_yaw, 0.0, -d_pitch)


@pytest.mark.parametrize("name,over,roll,pitch", SCENES)
def test_rolled_camera_equals_the_general_kernel(name, over, roll, pitch, monkeypatch):
    """A camera with roll: du.y != 0, the kernel computes the plane test per ray."""
    g = level_scene(name, over, roll, pitch)
    g.camera_rotate(0.0, 7.0, pitch)
    g.set_frame_size(333, 187)
    cam, _ = g.frame_blocks(seed=5)
    assert cam.up_left[1] != cam.up_right[1]
    assert_same_as_general(g, monkeypatch, f"{name} roll 7")


@pytest.mark.parametrize("compact", [0, 1])
@pytest.mark.parametrize("name,over,roll,pitch", SCENES)
def test_row_bands_equal_the_general_kernel(name, over, roll, pitch, compact, monkeypatch):
    """The table is built for the CTA's GLOBAL rows: 3 ranks' bands on one GPU, reassembled."""
    g = level_scene(name, over, roll, pitch)
    g.camera_rotate(0.0, 0.0, pitch)
    for w in (333, 330):
        g.set_frame_size(w, 187)
        camera_rows(g)
        (rgb, argb), (rgb_g, argb_g) = fast_and_general(monkeypatch, lambda: render_device_bands(g, 3, 16, compact))
        np.testing.assert_array_equal(rgb, rgb_g)
        np.testing.assert_array_equal(argb, argb_g)
        full, full_a, _ = g.render(argb=True, seed=5)
        np.testing.assert_array_equal(rgb, full)
        np.testing.assert_array_equal(argb, full_a)
