"""The one-plane frame kernel (render_kernel.cu render_solo_kernel: two adjacent pixels per thread, 32x8-pixel tiles, vector
stores straight to the frame) against the general kernel of the same scene class (C2RT_NO_SOLO_FAST=1, read per frame), where
its edges are: odd and even frame widths around the 32-pixel tiles, heights around the 8-row tiles, AA on and off, ARGB-only
delivery, row bands (full and compact), output planes off the vector alignment, and the ray counters.  The frames must be
BIT-identical."""
import os

import numpy as np
import pytest

import chess2rt_b200 as c2
from chess2rt_b200 import api, bands

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SC = os.path.join(ROOT, "scenes")

SCENES = [("lecture4-proc-texture.sdl", {}), ("lecture4.sdl", {}), ("../tests/scenes/sky_plane.sdl", {}), ("zaphod.sdl", {"dof": 0})]
WIDTHS = (1, 3, 4, 32, 33, 63, 64, 65, 66, 130, 333)
HEIGHTS = (1, 7, 9, 187)


@pytest.fixture(scope="module", autouse=True)
def _ctx():
    c2.init(1, [0])
    yield
    c2.shutdown()


def scene(name, over, aa):
    g = c2.HostScene(os.path.join(SC, name))
    g.override(aa=aa, **over)
    return g


def fast_and_general(monkeypatch, fn):
    monkeypatch.delenv("C2RT_NO_SOLO_FAST", raising=False)
    fast = fn()
    monkeypatch.setenv("C2RT_NO_SOLO_FAST", "1")
    general = fn()
    monkeypatch.delenv("C2RT_NO_SOLO_FAST")
    return fast, general


@pytest.mark.parametrize("aa", [1, 0])
@pytest.mark.parametrize("name,over", SCENES)
def test_tile_edges_equal_the_general_kernel(name, over, aa, monkeypatch):
    g = scene(name, over, aa)
    lit = 0.0
    for w in WIDTHS:
        for h in HEIGHTS:
            g.set_frame_size(w, h)
            (rgb, argb, st), (rgb_g, argb_g, st_g) = fast_and_general(monkeypatch, lambda: g.render(argb=True, seed=5, count_rays=True))
            what = f"{name} aa={aa} {w}x{h}"
            np.testing.assert_array_equal(rgb, rgb_g, err_msg=what)
            np.testing.assert_array_equal(argb, argb_g, err_msg=what)
            assert (st.primary_rays, st.shadow_rays) == (st_g.primary_rays, st_g.shadow_rays), what
            assert st.primary_rays == w * h * (5 if aa else 1), what
            lit = max(lit, float(rgb.max()))
    assert lit > 0.05


@pytest.mark.parametrize("name,over", SCENES)
def test_argb_only_delivery_equals_the_general_kernel(name, over, monkeypatch):
    g = scene(name, over, 1)
    for w, h in ((333, 187), (64, 9), (66, 7), (3, 1)):
        g.set_frame_size(w, h)
        (none, only, _), (_, only_g, _) = fast_and_general(monkeypatch, lambda: g.render(argb_only=True, seed=5))
        _, both_a, _ = g.render(argb=True, seed=5)
        assert none is None
        np.testing.assert_array_equal(only, only_g)
        np.testing.assert_array_equal(only, both_a)


def render_device_bands(g, n_ranks, band_rows, compact):
    """n ranks one after another on one GPU through c2rt_render_device, reassembled into the full frame."""
    import torch
    w, h = g.frame_size
    cam, st = g.frame_blocks(seed=5)
    handle = g.device_scene()
    stream = torch.cuda.current_stream().cuda_stream
    if not compact:
        frame = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
        argb = torch.zeros((h, w), dtype=torch.int32, device="cuda")
        for r in range(n_ranks):
            c2.render_device(handle, cam, st, frame.data_ptr(), argb.data_ptr(), api.Band(r, n_ranks, band_rows, 0), stream)
        torch.cuda.synchronize()
        return frame.cpu().numpy(), argb.cpu().numpy().view(np.uint32)
    pad = bands.rows_padded(h, n_ranks, band_rows)
    gathered = torch.zeros((n_ranks, pad, w, 3), dtype=torch.float32, device="cuda")
    gathered_a = torch.zeros((n_ranks, pad, w), dtype=torch.int32, device="cuda")
    for r in range(n_ranks):
        c2.render_device(handle, cam, st, gathered[r].data_ptr(), gathered_a[r].data_ptr(), api.Band(r, n_ranks, band_rows, 1), stream)
    frame = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
    argb = torch.empty((h, w), dtype=torch.int32, device="cuda")
    c2.deinterleave(gathered.data_ptr(), frame.data_ptr(), w, h, 3, n_ranks, band_rows, pad, stream)
    c2.deinterleave(gathered_a.data_ptr(), argb.data_ptr(), w, h, 1, n_ranks, band_rows, pad, stream)
    torch.cuda.synchronize()
    return frame.cpu().numpy(), argb.cpu().numpy().view(np.uint32)


def test_planes_four_bytes_off_alignment():
    """c2rt_render_device asks 16-byte alignment of d_rgb only when the width is a multiple of 4, and none of d_argb: at an
    even width with both planes 4 bytes off an 8-byte boundary the two-pixel vector stores must give way to scalar ones."""
    import torch
    g = scene("lecture4-proc-texture.sdl", {}, 1)
    g.set_frame_size(66, 9)
    full, full_a, _ = g.render(argb=True, seed=5)
    cam, st = g.frame_blocks(seed=5)
    rgb = torch.zeros(66 * 9 * 3 + 1, dtype=torch.float32, device="cuda")
    argb = torch.zeros(66 * 9 + 1, dtype=torch.int32, device="cuda")
    c2.render_device(g.device_scene(), cam, st, rgb.data_ptr() + 4, argb.data_ptr() + 4, None, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(rgb[1:].cpu().numpy().reshape(9, 66, 3), full)
    np.testing.assert_array_equal(argb[1:].cpu().numpy().view(np.uint32).reshape(9, 66), full_a)


@pytest.mark.parametrize("compact", [0, 1])
@pytest.mark.parametrize("name,over", SCENES)
def test_row_bands_equal_the_general_kernel(name, over, compact, monkeypatch):
    g = scene(name, over, 1)
    for w in (333, 330):   # odd (scalar stores) and even (vector stores) widths; 187 rows: the last band partial
        g.set_frame_size(w, 187)
        (rgb, argb), (rgb_g, argb_g) = fast_and_general(monkeypatch, lambda: render_device_bands(g, 3, 16, compact))
        np.testing.assert_array_equal(rgb, rgb_g)
        np.testing.assert_array_equal(argb, argb_g)
        full, full_a, _ = g.render(argb=True, seed=5)
        np.testing.assert_array_equal(rgb, full)
        np.testing.assert_array_equal(argb, full_a)
