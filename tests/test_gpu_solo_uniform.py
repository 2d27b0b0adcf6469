"""The straight-line tap of the one-plane frame kernel (render_kernel.cu render_solo_kernel<..., ROWS = true>, row_tap_settles,
light_far): a warp whose row-table entries settle every per-ray decision of the tap (plane hit, Procedure2 sine range, near-light
fallback, Lambert cosine) for both end columns of its tile row runs the tap without them.  Every frame must be BIT-identical to
the general kernel (C2RT_NO_SOLO_FAST=1), the ARGB plane and the ray counts included, and a numpy replay of the warp decision
must find warps on both loops in every frame: the horizon between the two rows of one warp, the Procedure2 bound crossing a tile
row, pixels under a low light, Checker and Phong frames at widths that are not multiples of 32, and row bands."""
import math
import os

import numpy as np
import pytest

import chess2rt_b200 as c2
from test_gpu_solo_rows import assert_same_as_general, camera_rows, level_scene
from test_gpu_solo_tiles import fast_and_general, render_device_bands

pytestmark = pytest.mark.gpu

KX, KY = (0.0, 0.3, 0.6, 0.0, 0.6), (0.0, 0.3, 0.0, 0.6, 0.6)   # AA tap offsets (renderer.d:235-242)
TILE_W, TILE_H, WARP_ROWS = 32, 8, 2                             # render_solo_kernel: a warp covers 2 rows of a 32x8 tile
MARGIN = 1e-6                                                    # relative: a replayed test this close to its bound is "unsure"

# floor height, light position, Procedure2 frequencies (rad / unit, U and V; None: no Procedure2) of each scene file
SCENES = {
    "lecture4-proc-texture.sdl": (2.0, (-30.0, 100.0, 250.0), ((0.01, 0.25, 0.01), (0.01, 0.25, 0.01))),
    "lecture4.sdl": (2.0, (-30.0, 100.0, 250.0), None),
    "../tests/scenes/proc_far.sdl": (-2.0, (-30.0, 120.0, 60.0), ((16470, 0.37, 16470), (0.02, 9100, 9100))),
    "../tests/scenes/proc_light_low.sdl": (2.0, (40.0, 5.0, 120.0), ((0.01, 0.25, 0.01), (0.01, 0.25, 0.01))),
    "../tests/scenes/phong_sharp.sdl": (0.0, (10.0, 60.0, 40.0), None),
}


@pytest.fixture(scope="module", autouse=True)
def _ctx():
    c2.init(1, [0])
    yield
    c2.shutdown()


def warp_paths(g, name):
    """Replays the warp vote in float64: counts of the warps that certainly take the straight-line tap, that certainly take the
    per-ray loop, and (reason -> count) of the latter."""
    plane_y, light, freqs = SCENES[name]
    cam, st = g.frame_blocks(seed=5)
    W, H = st.frame_width, st.frame_height
    pos = np.array(cam.pos)
    ul = np.array(cam.up_left) - pos
    du = np.array(cam.up_right) - np.array(cam.up_left)
    dv = np.array(cam.down_left) - np.array(cam.up_left)
    L = np.array(light)
    side = 1.0 if pos[1] > plane_y else -1.0
    near2 = 0.0576 * float(L @ L)
    lim = [2.0 ** 18 * 2 * math.pi / max(abs(f) for f in fr) for fr in freqs] if freqs else None
    dy_rows, graze_dy2 = camera_rows(g)
    n_tiles_y = (H + TILE_H - 1) // TILE_H
    uniform = general = 0
    why = {"horizon": 0, "sine range": 0, "near light": 0}
    for ty in range(n_tiles_y):
        for w in range(TILE_H // WARP_ROWS):
            rows = [ty * TILE_H + w * WARP_ROWS + i for i in range(WARP_ROWS)]
            if rows[0] >= H:
                continue
            for tx in range((W + TILE_W - 1) // TILE_W):
                ends = (tx * TILE_W, min(tx * TILE_W + TILE_W - 1, W - 1))
                sure_no, unsure = set(), False
                for y in rows:
                    for k in range(5):
                        sy = (y + KY[k]) / cam.frame_height
                        dy = dy_rows[y, k] if y < H else ul[1] + dv[1] * sy
                        if dy * dy < 4 * graze_dy2:   # at the grazing prefilter or the sign test's edge
                            unsure = True
                            continue
                        if dy * side > 0:             # d.y points away from the plane: ROW_MISS
                            sure_no.add("horizon")
                            continue
                        t = -(pos[1] - plane_y) / dy
                        fD = []
                        for x in ends:
                            sx = (x + KX[k]) / cam.frame_width
                            d = ul + du * sx + dv * sy
                            p = pos + d * t
                            if lim:
                                r = max(abs(p[0]) / lim[0], abs(p[2]) / lim[1])
                                if r > 1 + MARGIN:
                                    sure_no.add("sine range")
                                elif r > 1 - MARGIN:
                                    unsure = True
                            fD.append((L[0] - p[0], L[2] - p[2]))
                        (xa, za), (xb, zb) = fD
                        mx = min(abs(xa), abs(xb)) if (xa > 0) == (xb > 0) else 0.0
                        mz = min(abs(za), abs(zb)) if (za > 0) == (zb > 0) else 0.0
                        fDy = L[1] - plane_y - side * 1e-6
                        d2 = mx * mx + fDy * fDy + mz * mz
                        if d2 < near2 * (1 - MARGIN):
                            sure_no.add("near light")
                        elif d2 < near2 * (1 + MARGIN):
                            unsure = True
                if sure_no:
                    general += 1
                    for r in sure_no:
                        why[r] += 1
                elif not unsure:
                    uniform += 1
    return uniform, general, why


def check_frame(g, name, monkeypatch, what, reason):
    uniform, general, why = warp_paths(g, name)
    assert uniform > 0 and why[reason] > 0, (what, uniform, general, why)
    assert_same_as_general(g, monkeypatch, what)
    return why


def test_horizon_between_the_two_rows_of_a_warp(monkeypatch):
    """A level camera pitched up until the horizon falls between the rows of one warp: the row above misses the plane in every
    tap, the row below hits it in every tap."""
    name = "lecture4-proc-texture.sdl"
    g = level_scene(name, {}, 0.0, -30.0)
    g.set_frame_size(333, 187)
    found = 0
    for step in range(1, 400):
        g.camera_rotate(0.0, 0.0, 0.05)
        dy, _ = camera_rows(g)
        miss = ~np.signbit(dy)
        split = [y for y in range(0, dy.shape[0] - 1, WARP_ROWS) if miss[y].all() and not miss[y + 1].any()]
        if split:
            found += 1
            check_frame(g, name, monkeypatch, f"pitch {0.05 * step:.2f} horizon below row {split[0]}", "horizon")
            if found == 3:
                break
    assert found == 3


@pytest.mark.parametrize("yaw", [0.0, 23.0, -61.0])
def test_procedure2_bound_inside_a_tile_row(yaw, monkeypatch):
    """proc_far without its roll: the fast sine's range ends inside the frame; with a yaw its boundary crosses tile rows, so a
    warp can have one end column inside the range and the other outside."""
    name = "../tests/scenes/proc_far.sdl"
    g = level_scene(name, {}, 2.0, -45.0)
    g.camera_rotate(yaw, 0.0, -45.0)
    for w, h in ((203, 131), (333, 187)):
        g.set_frame_size(w, h)
        check_frame(g, name, monkeypatch, f"proc_far yaw {yaw} {w}x{h}", "sine range")


@pytest.mark.parametrize("yaw", [0.0, 15.0])
def test_pixels_under_a_low_light(yaw, monkeypatch):
    name = "../tests/scenes/proc_light_low.sdl"
    g = level_scene(name, {}, 0.0, -30.0)
    g.camera_rotate(yaw, 0.0, -30.0)
    for w, h in ((320, 240), (333, 187), (65, 41)):
        g.set_frame_size(w, h)
        check_frame(g, name, monkeypatch, f"proc_light_low yaw {yaw} {w}x{h}", "near light")


@pytest.mark.parametrize("name", ["lecture4.sdl", "../tests/scenes/phong_sharp.sdl", "lecture4-proc-texture.sdl"])
def test_checker_phong_and_ragged_widths(name, monkeypatch):
    """The horizon in the frame (warps above it take the per-ray loop) at widths whose last tile row is clamped to W - 1."""
    g = level_scene(name, {}, 0.0, -30.0)
    g.camera_rotate(17.0, 0.0, 6.0)
    for w, h in ((333, 187), (65, 41), (97, 64), (31, 17)):
        g.set_frame_size(w, h)
        check_frame(g, name, monkeypatch, f"{name} {w}x{h}", "horizon")


@pytest.mark.parametrize("compact", [0, 1])
@pytest.mark.parametrize("name", ["lecture4-proc-texture.sdl", "../tests/scenes/proc_light_low.sdl"])
def test_row_bands(name, compact, monkeypatch):
    """3 ranks' bands on one GPU, reassembled: the warp decision is taken on the CTA's global rows."""
    g = level_scene(name, {}, 0.0, -30.0)
    g.camera_rotate(9.0, 0.0, 6.0 if name == "lecture4-proc-texture.sdl" else -30.0)
    for w in (333, 330):
        g.set_frame_size(w, 187)
        uniform, general, why = warp_paths(g, name)
        assert uniform > 0 and general > 0, (uniform, general, why)
        (rgb, argb), (rgb_g, argb_g) = fast_and_general(monkeypatch, lambda: render_device_bands(g, 3, 16, compact))
        np.testing.assert_array_equal(rgb, rgb_g)
        np.testing.assert_array_equal(argb, argb_g)
        full, full_a, _ = g.render(argb=True, seed=5)
        np.testing.assert_array_equal(rgb, full)
        np.testing.assert_array_equal(argb, full_a)
