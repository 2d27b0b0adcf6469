"""Parity tests proper: the CUDA path, called through the C ABI (libc2rt.so via the host mirror),
against the CPU oracle on the same inputs.  Bar (BASELINE.json north_star): per-pixel float RGB within
1e-3 absolute; at most 0.1 % of 8-bit pixels differing by more than 1 LSB.  Integer work (ARGB packing,
ray counts, band scatter) must be bit-exact."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import chess2rt_b200 as c2
from chess2rt_b200 import api, bands
from oracle_binding import OracleScene, pack_rgb32, parity_report

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SC = os.path.join(ROOT, "scenes")
GOLD = os.path.join(ROOT, "tests", "golden")
TOL = 1e-3  # float RGB, absolute (north_star)


@pytest.fixture(scope="module", autouse=True)
def _ctx():
    c2.init(1, [0])
    yield
    c2.shutdown()


def both(path, size=None, seed=0, **over):
    g, o = c2.HostScene(path), OracleScene(path)
    for s in (g, o):
        if size:
            s.set_frame_size(*size)
        s.override(**over)
    return g, o


def assert_parity(rgb, ref, argb=None, what=""):
    rep = parity_report(rgb, ref, argb)
    assert rep["px_over_1e-3"] == 0, (what, rep)
    assert rep["frac_over_1lsb"] <= 1e-3, (what, rep)
    return rep


CASES = [
    ("lecture4.sdl", None, {}),
    ("lecture4.json", None, {}),
    ("lecture4-proc-texture.sdl", None, {}),
    ("lecture5.sdl", None, {}),
    ("zaphod.sdl", None, {"dof": 0}),          # 645x430: not a multiple of the 16x8 tile nor of 4
    ("zaphod.sdl", None, {"num_samples": 6}),  # DOF with the pinned generator
    ("chessboard.sdl", (480, 270), {}),
    ("../tests/scenes/quirks.sdl", None, {}),
    ("../tests/scenes/nested.sdl", None, {}),   # CSG inside CSG: literal emulation path
    ("../tests/scenes/stereo.sdl", None, {}),       # anaglyph stereo: two eyes per sample, combineStereo
    ("../tests/scenes/stereo_dof.sdl", None, {}),   # stereo + DOF: each eye draws its own jitter and lens sample
    ("../tests/scenes/sky.sdl", None, {}),          # cubemap-environment EXTENSION: misses sample the sky faces (warp-mask kernels)
    ("../tests/scenes/sky_plane.sdl", None, {}),    # the same on the one-plane scene class (MODE_SOLO kernels), assumedGamma 1.8
    ("../tests/scenes/sky.sdl", (97, 61), {"aa": 0}),
    ("zaphod-sky.sdl", (215, 143), {"num_samples": 4}),   # configs[3] "with cubemap skybox": DOF over the page, sky behind the camera
    ("../tests/scenes/proc_far.sdl", None, {}),       # Procedure2: fast one-step sine reduction and its far-distance fallback in one frame, shared sines
    ("../tests/scenes/proc_far.sdl", None, {"aa": 0}),
    ("../tests/scenes/proc_below.sdl", None, {}),     # one-plane class from below the plane, Phong lobe, three equal frequencies
    ("../tests/scenes/proc_inplane.sdl", None, {}),   # camera in the plane: the fixed-side shortcut must stand aside
]


@pytest.mark.parametrize("name,size,over", CASES)
def test_scene_matches_oracle(name, size, over):
    g, o = both(os.path.join(SC, name), size, **over)
    rgb, argb, st = g.render(argb=True, seed=11, count_rays=True)
    ref, ost = o.render(seed=11)
    assert_parity(rgb, ref, argb, name)
    # rays the algorithm requires: identical counts (same hit / lit decisions)
    assert (st.primary_rays, st.shadow_rays) == (ost.primary_rays, ost.shadow_rays)
    # ARGB plane == Color.toRGB32 of the float plane, bit-exact
    np.testing.assert_array_equal(argb, pack_rgb32(rgb))
    assert ost.csg_max_crossings <= 8  # the nested-CSG path's per-child crossing capacity


@pytest.mark.parametrize("name,size", [("../tests/scenes/quirks.sdl", None), ("chessboard.sdl", (320, 180)), ("lecture5.sdl", (320, 240))])
def test_closed_form_csg_equals_literal_walk(name, size, monkeypatch):
    """The register-only closed-form CSG and the literal replay of the reference's restart/sort/walk agree."""
    g, o = both(os.path.join(SC, name), size)
    fast, _, st_fast = g.render(count_rays=True)
    monkeypatch.setenv("C2RT_CSG_LITERAL", "1")   # read at scene-create time
    lit_scene = c2.HostScene(os.path.join(SC, name))
    if size:
        lit_scene.set_frame_size(*size)
    lit, _, st_lit = lit_scene.render(count_rays=True)
    ref, ost = o.render()
    assert_parity(lit, ref, what="literal " + name)
    assert_parity(fast, ref, what="closed form " + name)
    assert (st_lit.primary_rays, st_lit.shadow_rays) == (st_fast.primary_rays, st_fast.shadow_rays) == (ost.primary_rays, ost.shadow_rays)
    assert np.abs(fast - lit).max() < 1e-5


SOLO_SCENE = """Scene {{
  GlobalSettings {{ frameWidth 322; frameHeight 203; ambientLightColor 0.03 0.02 0.04; prepassEnabled false }}
  Camera {{ pos 3 {camy} -20; yaw 12; pitch {pitch}; roll 4; fov 80{cam_extra} }}
  Lights {{ PointLight "l" {{ pos -40 {lighty} 90; color 1 0.9 0.8; power 30000 }} }}
  Geometries {{ Plane "floor" {{ y 1.5 }} }}
  Textures {{
    Checker "decoy" {{ color1 1 0 0; color2 0 1 0; size 2 }}
    BitmapTexture "decoy2" {{ file "{root}/scenes/world.bmp" }}
    Checker "chk" {{ color1 0.1 0.2 0.1; color2 0.9 0.6 0.2; size 7 }}
    Procedure2 "proc" {{
      freqU 0.3 0.11 0.05
      freqV 0.07 0.4 0.13
      colorU {{ color 0.4 0.1 0.2; color 0.2 0.3 0.1; color 0.1 0.2 0.4 }}
      colorV {{ color 0.1 0.3 0.3; color 0.3 0.1 0.1; color 0.2 0.2 0.2 }}
    }}
    BitmapTexture "bmp" {{ file "{root}/scenes/floor.bmp"; scaling 0.02; assumedGamma 1.8 }}
  }}
  Shaders {{
    Lambert "decoy_shader" {{ color 0 0 1; texture "decoy" }}
    Phong "decoy_shader2" {{ color 0 1 1; exponent 5 }}
    {shader} "s" {{ color 0.7 0.5 0.3{tex}{shader_extra} }}
  }}
  Nodes {{ Node "n" {{ geometry "floor"; shader "s"{node_extra} }} }}
}}
"""


@pytest.mark.parametrize("shader", ["Lambert", "Phong"])
@pytest.mark.parametrize("tex", [None, "chk", "proc", "bmp"])
@pytest.mark.parametrize("variant", ["plain", "below_scaled", "dof"])
def test_solo_scene_class_kernels(shader, tex, variant, tmp_path, monkeypatch):
    """One plane + one light scenes run on the MODE_SOLO kernels (scene constants at static addresses, texture and shader
    kind compiled in; the node's shader / texture are moved to record 0 at scene create).  Each of the 8 kinds, with and
    without the sampling loop, against the oracle and against the general plane-only kernel (C2RT_NO_SOLO=1)."""
    text = SOLO_SCENE.format(
        root=ROOT, shader=shader, tex=f'; texture "{tex}"' if tex else "",
        shader_extra="; exponent 24; strength 0.8" if shader == "Phong" else "",
        camy=-60 if variant == "below_scaled" else 45, pitch=25 if variant == "below_scaled" else -22,
        lighty=-80 if variant == "below_scaled" else 70,    # camera and light under the plane: the face-forward flip
        node_extra="; scale 3 2 0.5; translate 4 1 -6" if variant == "below_scaled" else "",
        cam_extra="; dof true; numSamples 3; focalPlaneDist 60; fNumber 4" if variant == "dof" else "")
    path = tmp_path / "solo.sdl"
    path.write_text(text)
    g, o = both(str(path))
    rgb, argb, st = g.render(argb=True, seed=5, count_rays=True)
    ref, ost = o.render(seed=5)
    assert ref.max() > 0.05
    assert_parity(rgb, ref, argb, f"solo {shader} {tex} {variant}")
    assert (st.primary_rays, st.shadow_rays) == (ost.primary_rays, ost.shadow_rays)
    monkeypatch.setenv("C2RT_NO_SOLO", "1")   # read at scene-create time
    general = c2.HostScene(str(path))
    rgb2, _, st2 = general.render(seed=5, count_rays=True)
    assert (st2.primary_rays, st2.shadow_rays) == (st.primary_rays, st.shadow_rays)
    assert np.abs(rgb - rgb2).max() < 1e-5


@pytest.mark.parametrize("name,size,over", [("zaphod.sdl", (322, 214), {"num_samples": 3}), ("lecture5.sdl", (330, 203), {}),
                                            ("zaphod.sdl", (160, 90), {"dof": 0})])
def test_palette_quad_bitmaps_equal_float4_texels(name, size, over, monkeypatch):
    """Bitmaps with <= 256 distinct colours are stored as palette-index quads (one 4-byte load per bilinear lookup,
    scene_dev.h DevTex::quads): the frame must be BIT-identical to the float4-texel form (C2RT_NO_PALETTE=1)."""
    g = c2.HostScene(os.path.join(SC, name))
    g.set_frame_size(*size)
    g.override(**over)
    pal, pal_a, _ = g.render(argb=True, seed=7)
    monkeypatch.setenv("C2RT_NO_PALETTE", "1")   # read at scene-create time
    h = c2.HostScene(os.path.join(SC, name))
    h.set_frame_size(*size)
    h.override(**over)
    flt, flt_a, _ = h.render(argb=True, seed=7)
    np.testing.assert_array_equal(pal, flt)
    np.testing.assert_array_equal(pal_a, flt_a)
    assert pal.max() > 0.05


@pytest.mark.parametrize("name,size,over", [("lecture4-proc-texture.sdl", (333, 187), {}), ("lecture4.sdl", None, {}),
                                            ("../tests/scenes/proc_below.sdl", None, {}), ("../tests/scenes/proc_far.sdl", None, {}),
                                            ("../tests/scenes/sky_plane.sdl", None, {}), ("zaphod.sdl", (161, 107), {"dof": 0}),
                                            ("zaphod.sdl", (161, 107), {"num_samples": 3})])   # DOF: the whole lens is checked
def test_regular_one_plane_frames_equal_the_general_kernel(name, size, over, monkeypatch):
    """One-plane frames with a fixed camera off the plane and the light on its side run on kernels that take the camera's
    side, its height and 'the plane cannot shadow itself' as frame constants (render_kernel.cu solo_plane_test, c2rt_api.cu
    fill_params).  Those are shortcuts, not approximations: the frame must be BIT-identical to the one the general kernel of
    the scene class renders (C2RT_NO_SOLO_FAST=1, read per frame), ray counts included."""
    g = c2.HostScene(os.path.join(SC, name))
    if size:
        g.set_frame_size(*size)
    g.override(**over)
    fast, fast_a, st_fast = g.render(argb=True, seed=5, count_rays=True)
    monkeypatch.setenv("C2RT_NO_SOLO_FAST", "1")
    gen, gen_a, st_gen = g.render(argb=True, seed=5, count_rays=True)
    np.testing.assert_array_equal(fast, gen)
    np.testing.assert_array_equal(fast_a, gen_a)
    assert (st_fast.primary_rays, st_fast.shadow_rays) == (st_gen.primary_rays, st_gen.shadow_rays)
    assert fast.max() > 0.05


def test_cubemap_extension_is_inert_where_no_ray_misses_and_refuses_gi(tmp_path):
    """zaphod-sky.sdl = zaphod.sdl + the cubemap environment: its camera looks down at the page, no ray misses, so the frame is
    bit-identical to zaphod.sdl's.  GI frames are only built for the reference's black environment: refused with a cubemap."""
    a = c2.HostScene(os.path.join(SC, "zaphod.sdl"))
    b = c2.HostScene(os.path.join(SC, "zaphod-sky.sdl"))
    for s in (a, b):
        s.set_frame_size(200, 133)
        s.override(num_samples=3)
    np.testing.assert_array_equal(a.render(seed=4)[0], b.render(seed=4)[0])
    txt = open(os.path.join(ROOT, "tests", "scenes", "sky.sdl")).read()
    txt = txt.replace('"../../scenes/skybox"', '"%s/skybox"' % SC).replace("AAEnabled true", "AAEnabled true\n    GIEnabled true")
    txt = txt.replace('Phong "shiny" { color 0.8 0.3 0.2; exponent 40; strength 0.7 }', 'Lambert "shiny" { color 0.8 0.3 0.2 }')
    p = tmp_path / "gi_sky.sdl"
    p.write_text(txt)
    with pytest.raises(c2.C2rtError, match="cubemap"):
        c2.HostScene(str(p)).render()


def test_golden_fixtures():
    meta = json.load(open(os.path.join(GOLD, "golden.json")))
    for name, m in meta.items():
        g = c2.HostScene(os.path.join(ROOT, m["scene"]))
        g.set_frame_size(*m["size"])
        g.override(**m["override"])
        rgb, _, st = g.render(seed=m["seed"], count_rays=True)
        assert_parity(rgb, np.load(os.path.join(GOLD, name + ".npy")), what=name)
        assert (st.primary_rays, st.shadow_rays) == (m["primary_rays"], m["shadow_rays"])


def test_config_c1_1080p_full_frame():
    # BASELINE.json configs[1]: lecture4-proc-texture.sdl at 1920x1080
    g, o = both(os.path.join(SC, "lecture4-proc-texture.sdl"), (1920, 1080))
    rgb, argb, st = g.render(argb=True, count_rays=True)
    ref, ost = o.render()
    assert_parity(rgb, ref, argb, "C1")
    assert st.primary_rays == 1920 * 1080 * 5 and st.shadow_rays == ost.shadow_rays


def test_config_c2_4k_row_windows():
    # configs[2]: lecture5.sdl at 3840x2160 — full GPU frame, oracle on row windows spread over the frame
    g, o = both(os.path.join(SC, "lecture5.sdl"), (3840, 2160))
    rgb, _, _ = g.render()
    for y0 in (0, 400, 777, 1200, 1650, 2144):
        ref, _ = o.render_rows(y0, y0 + 16)
        assert_parity(rgb[y0:y0 + 16], ref, what=f"C2 rows {y0}")


def test_config_c3_zaphod_4k_dof_windows():
    # configs[3]: zaphod.sdl at 3840x2160 with DOF (25 samples x 5 taps), pinned RNG, "with cubemap skybox": the reference has no
    # cubemap (SURVEY F3); zaphod-sky.sdl adds the extension's environment block
    g, o = both(os.path.join(SC, "zaphod-sky.sdl"), (3840, 2160))
    rgb, _, _ = g.render(seed=99)
    for y0 in (8, 1080, 2150):
        ref, _ = o.render_rows(y0, y0 + 4, seed=99)
        assert_parity(rgb[y0:y0 + 4], ref, what=f"C3 rows {y0}")


def test_config_c4_chessboard_8k_windows_and_properties():
    # configs[4]: synthetic chessboard at 7680x4320 — oracle on row windows + size-independent properties
    g, o = both(os.path.join(SC, "chessboard.sdl"), (7680, 4320))
    rgb, argb, st = g.render(argb=True, count_rays=True)
    for y0 in (0, 1500, 2800, 3600, 4312):
        ref, _ = o.render_rows(y0, y0 + 8)
        assert_parity(rgb[y0:y0 + 8], ref, what=f"C4 rows {y0}")
    assert st.primary_rays == 7680 * 4320 * 5
    assert st.shadow_rays == st.primary_rays        # every primary ray hits (floor fills the view), one live light
    np.testing.assert_array_equal(argb, pack_rgb32(rgb))
    assert np.isfinite(rgb).all() and rgb.min() >= 0
    # idempotence: the frame is a pure function of (scene, camera, settings)
    rgb2, _, _ = g.render()
    np.testing.assert_array_equal(rgb, rgb2)


@pytest.mark.parametrize("size", [(1, 1), (3, 2), (17, 9), (16, 8), (33, 41), (130, 7)])
def test_ragged_and_tiny_frames(size):
    g, o = both(os.path.join(SC, "lecture5.sdl"), size)
    rgb, argb, _ = g.render(argb=True)
    ref, _ = o.render()
    assert rgb.shape == (size[1], size[0], 3)
    assert_parity(rgb, ref, argb, str(size))


def test_render_pixel_matches_oracle_hit_record():
    path = os.path.join(ROOT, "tests", "scenes", "quirks.sdl")
    g, o = both(path)
    for (x, y) in [(10, 10), (160, 100), (60, 120), (200, 110), (250, 120), (300, 180), (120, 60), (90, 150), (0, 0)]:
        rgb, hit = g.render_pixel(x, y)
        ref_rgb, ref_hit = o.render_pixel(x, y)
        assert hit.node == int(ref_hit[0]), (x, y)
        np.testing.assert_allclose(rgb, ref_rgb, atol=TOL)
        if hit.node >= 0:
            np.testing.assert_allclose(hit.dist, ref_hit[1], rtol=1e-12)
            np.testing.assert_allclose(list(hit.p), ref_hit[2:5], rtol=1e-11, atol=1e-9)
            np.testing.assert_allclose(list(hit.normal), ref_hit[5:8], atol=1e-12)
            np.testing.assert_allclose([hit.u, hit.v], ref_hit[8:10], rtol=1e-10, atol=1e-9)


def _render_device_bands(g, n_ranks, band_rows, compact, seed=0):
    """Emulates n ranks one after another on one GPU through c2rt_render_device (no waiting between kernels)."""
    import torch
    w, h = g.frame_size
    cam, st = g.frame_blocks(seed=seed)
    handle = g.device_scene()
    if not compact:
        frame = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
        argb = torch.zeros((h, w), dtype=torch.int32, device="cuda")
        for r in range(n_ranks):
            band = api.Band(r, n_ranks, band_rows, 0)
            c2.render_device(handle, cam, st, frame.data_ptr(), argb.data_ptr(), band, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        return frame.cpu().numpy(), argb.cpu().numpy().view(np.uint32)
    pad = bands.rows_padded(h, n_ranks, band_rows)
    gathered = torch.zeros((n_ranks, pad, w, 3), dtype=torch.float32, device="cuda")
    gathered_a = torch.zeros((n_ranks, pad, w), dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    for r in range(n_ranks):
        band = api.Band(r, n_ranks, band_rows, 1)
        c2.render_device(handle, cam, st, gathered[r].data_ptr(), gathered_a[r].data_ptr(), band, stream)
    frame = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
    argb = torch.empty((h, w), dtype=torch.int32, device="cuda")
    c2.deinterleave(gathered.data_ptr(), frame.data_ptr(), w, h, 3, n_ranks, band_rows, pad, stream)
    c2.deinterleave(gathered_a.data_ptr(), argb.data_ptr(), w, h, 1, n_ranks, band_rows, pad, stream)
    torch.cuda.synchronize()
    return frame.cpu().numpy(), argb.cpu().numpy().view(np.uint32)


@pytest.mark.parametrize("n_ranks,band_rows,compact", [(1, 8, 0), (2, 8, 0), (2, 8, 1), (3, 16, 1), (8, 8, 1), (4, 24, 0)])
def test_row_bands_reassemble_bit_exactly(n_ranks, band_rows, compact):
    g = c2.HostScene(os.path.join(SC, "lecture5.sdl"))
    g.set_frame_size(330, 203)   # ragged in x and y, last band partial
    full, full_a, _ = g.render(argb=True)
    rgb, argb = _render_device_bands(g, n_ranks, band_rows, compact)
    np.testing.assert_array_equal(rgb, full)
    np.testing.assert_array_equal(argb, full_a)


def test_ray_counters_device_path():
    g, o = both(os.path.join(SC, "lecture5.sdl"), (200, 120))
    import torch
    cam, st = g.frame_blocks(count_rays=True)
    frame = torch.zeros((120, 200, 3), dtype=torch.float32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    c2.render_device(g.device_scene(), cam, st, frame.data_ptr(), None, None, stream)
    p, s = c2.read_ray_counters(g.device_scene(), stream)
    _, ost = o.render()
    assert (p, s) == (ost.primary_rays, ost.shadow_rays)
    assert c2.read_ray_counters(g.device_scene(), stream) == (0, 0)


def test_gi_frames(tmp_path):
    """GIEnabled (renderer.d:260-263,289-301): black like the literal oracle walk; Phong scenes are refused (the reference
    halts in Phong.spawnRay); under DOF the GI flag is ignored."""
    from test_oracle_kat import GI_SCENE
    p = tmp_path / "gi.sdl"
    p.write_text(GI_SCENE.format(paths=3, cam="", ball_shader="Lambert"))
    g, o = both(str(p))
    rgb, argb, _ = g.render(argb=True, seed=2)
    ref, _ = o.render(seed=2)
    np.testing.assert_array_equal(rgb, ref)
    assert not rgb.any() and not argb.any()
    p.write_text(GI_SCENE.format(paths=0, cam="", ball_shader="Lambert"))
    assert np.all(np.isnan(c2.HostScene(str(p)).render()[0]))
    p.write_text(GI_SCENE.format(paths=3, cam="", ball_shader="Phong"))
    with pytest.raises(c2.C2rtError, match="Phong"):
        c2.HostScene(str(p)).render()
    p.write_text(GI_SCENE.format(paths=3, cam="; dof true; numSamples 2; focalPlaneDist 120; fNumber 8", ball_shader="Phong"))
    g, o = both(str(p))
    rgb, _, st = g.render(seed=3, count_rays=True)
    ref, ost = o.render(seed=3)
    assert_parity(rgb, ref, what="GI flag under DOF")
    assert (st.primary_rays, st.shadow_rays) == (ost.primary_rays, ost.shadow_rays)


def test_unsupported_features_are_errors_not_fallbacks():
    g = c2.HostScene(os.path.join(SC, "lecture5.sdl"))   # has Phong-shaded nodes
    cam, st = g.frame_blocks()
    rgb = np.zeros((480, 640, 3), np.float32)
    st.gi_enabled = 1
    assert api.lib.c2rt_render(g.device_scene(), C.byref(cam), C.byref(st), rgb.ctypes.data, None, None) == -2
    assert api.lib.c2rt_render_pixel(g.device_scene(), C.byref(cam), C.byref(st), 3, 3, (C.c_float * 3)(), None) == -2
    st.gi_enabled = 0
    assert api.lib.c2rt_render(g.device_scene(), C.byref(cam), C.byref(st), None, None, None) == -1
    assert api.lib.c2rt_render(g.device_scene(), C.byref(cam), C.byref(st), rgb.ctypes.data, None, None) == 0


@pytest.mark.parametrize("scene,size,extra", [("lecture5.sdl", (200, 150), ""), ("lecture5.sdl", (97, 61), "bucketSize 40"),
                                              ("zaphod.sdl", (130, 70), "")])
def test_prepass_only_preview(scene, size, extra, tmp_path):
    """prepassOnly (renderer.d:110-130): one sample per 16x16 block laid out inside each bucket, replicated."""
    txt = open(os.path.join(SC, scene)).read()
    txt = txt.replace('"floor.bmp"', '"%s/floor.bmp"' % SC).replace('"world.bmp"', '"%s/world.bmp"' % SC)
    txt = txt.replace('"texture/zaphod.bmp"', '"%s/texture/zaphod.bmp"' % SC)
    txt = txt.replace("prepassOnly         false", "").replace("prepassEnabled      false", "")
    txt = txt.replace("GlobalSettings {", "GlobalSettings {\n    prepassOnly true\n    prepassEnabled true\n    %s\n" % extra, 1)
    p = tmp_path / "prepass.sdl"
    p.write_text(txt)
    g, o = both(p, size)
    rgb, argb, _ = g.render(argb=True, seed=5)
    ref, _ = o.render(seed=5)
    assert_parity(rgb, ref, argb, "prepassOnly " + scene)
    # blocks really are constant
    assert np.array_equal(rgb[0:8, 0:16], np.broadcast_to(rgb[0, 0], (8, 16, 3)))
    # prepassOnly without prepassEnabled draws nothing: the caller's buffer keeps its contents
    p2 = tmp_path / "nothing.sdl"
    p2.write_text(txt.replace("prepassEnabled true", "prepassEnabled false"))
    g2 = c2.HostScene(p2)
    g2.set_frame_size(*size)
    buf = np.full((size[1], size[0], 3), 7.0, np.float32)
    g2.render(out=buf)
    assert (buf == 7.0).all()


def test_degenerate_scenes(tmp_path):
    """Empty node list, no lights, only a dark light, camera inside a CSG solid: still the oracle's image."""
    cases = {
        "empty": 'Scene { GlobalSettings { frameWidth 40; frameHeight 24 }\n Camera { pos 0 10 0; fov 90 } }',
        "nolights": 'Scene { GlobalSettings { frameWidth 40; frameHeight 24; ambientLightColor 0.3 0.2 0.1 }\n Camera { pos 0 50 -80; pitch -20; fov 80 }\n'
                    ' Geometries { Plane "f" { y 0 }; Sphere "s" { center 0 20 0; R 20 } }\n Shaders { Lambert "a" { color 1 0.5 0.25 } }\n'
                    ' Nodes { Node "n0" { geometry "f"; shader "a" }; Node "n1" { geometry "s"; shader "a" } } }',
        "darklight": 'Scene { GlobalSettings { frameWidth 40; frameHeight 24; ambientLightColor 0.1 0.1 0.1 }\n Camera { pos 0 50 -80; pitch -20; fov 80 }\n'
                     ' Lights { PointLight "l" { pos 0 100 0; color 1 1 1; power 0 } }\n'
                     ' Geometries { Plane "f" { y 0 } }\n Shaders { Phong "a" { color 1 0.5 0.25; exponent 10 } }\n Nodes { Node "n0" { geometry "f"; shader "a" } } }',
        "inside": 'Scene { GlobalSettings { frameWidth 48; frameHeight 32; ambientLightColor 0.05 0.05 0.05 }\n Camera { pos 0 0 0; yaw 20; pitch 10; fov 100 }\n'
                  ' Lights { PointLight "l" { pos 5 6 -4; color 1 1 1; power 900 } }\n'
                  ' Geometries { Cube "c" { side 60 }; Sphere "s" { R 36 }; CsgInter "i" { left "c"; right "s" }; CsgDiff "d" { left "s"; right "c" } }\n'
                  ' Shaders { Phong "a" { color 0.6 0.7 0.8; exponent 20 }; Lambert "b" { color 0.9 0.3 0.3 } }\n'
                  ' Nodes { Node "n0" { geometry "i"; shader "a" }; Node "n1" { geometry "d"; shader "b"; scale 1.5 1.5 1.5 } } }',
    }
    for name, txt in cases.items():
        p = tmp_path / (name + ".sdl")
        p.write_text(txt)
        g, o = both(p)
        rgb, argb, st = g.render(argb=True, count_rays=True)
        ref, ost = o.render()
        assert_parity(rgb, ref, argb, name)
        assert (st.primary_rays, st.shadow_rays) == (ost.primary_rays, ost.shadow_rays), name
    assert np.all(c2.HostScene(tmp_path / "empty.sdl").render()[0] == 0)


def big_scene_text(n_side, width=160, height=100):
    """n_side x n_side pieces (spheres, cubes, a CSG of both, every third one scaled) on a checker floor: n_side^2 + 1 nodes."""
    geoms = ['Plane "floor" { y 0 }', 'Sphere "s" { center 0 0 0; R 4 }', 'Cube "c" { center 0 0 0; side 7 }',
             'Sphere "cut" { center 2 2 -2; R 3.5 }', 'CsgDiff "d" { left "c"; right "cut" }', 'CsgUnion "u" { left "s"; right "c" }']
    nodes = ['Node "floor" { geometry "floor"; shader "f" }']
    k = 0
    for i in range(n_side):
        for j in range(n_side):
            g = ("s", "c", "d", "u")[k % 4]
            sh = ("a", "b", "p")[k % 3]
            scale = "scale 1.3 0.8 1.1; " if k % 3 == 0 else ""
            nodes.append('Node "n%d" { geometry "%s"; shader "%s"; %stranslate %g %g %g }' % (k, g, sh, scale, (i - n_side / 2) * 12.0, 4.0 + (k % 5), (j - n_side / 2) * 12.0))
            k += 1
    return ('Scene { GlobalSettings { frameWidth %d; frameHeight %d; ambientLightColor 0.1 0.1 0.12; AAEnabled true; prepassEnabled false }\n'
            ' Camera { pos 5 %g %g; yaw 8; pitch -32; roll 2; fov 70 }\n'
            ' Lights { PointLight "l" { pos -150 260 -120; color 1 0.95 0.9; power 70000 }; PointLight "l2" { pos 200 120 150; color 0.4 0.5 0.9; power 30000 } }\n'
            ' Geometries { %s }\n Textures { Checker "chk" { color1 0.15 0.15 0.2; color2 0.9 0.85 0.8; size 9 } }\n'
            ' Shaders { Lambert "f" { color 1 1 1; texture "chk" }; Lambert "a" { color 0.8 0.4 0.3 }; Lambert "b" { color 0.3 0.7 0.4 }; Phong "p" { color 0.3 0.4 0.9; exponent 30; strength 0.6 } }\n'
            ' Nodes { %s } }\n') % (width, height, 9.0 * n_side, -10.0 * n_side, "; ".join(geoms), "; ".join(nodes))


def test_scene_beyond_the_constant_block_renders_in_parity(tmp_path):
    """The reference's scene.nodes is unbounded (scene.d:38-51, renderer.d:336-338).  A scene beyond the constant block (64 nodes)
    keeps its records in global memory and walks multi-word node masks (MODE_BIG): 257 nodes, in parity with the oracle."""
    p = tmp_path / "big.sdl"
    p.write_text(big_scene_text(16))
    g, o = both(str(p))
    assert g.info()["nodes"] == 257
    rgb, argb, st = g.render(argb=True, count_rays=True)
    ref, ost = o.render()
    assert_parity(rgb, ref, argb, "257 nodes")
    assert (st.primary_rays, st.shadow_rays) == (ost.primary_rays, ost.shadow_rays)
    for (x, y) in [(80, 50), (20, 70), (140, 30), (0, 0)]:   # the pixel pick runs its own (one-warp) kernel
        c, hit = g.render_pixel(x, y)
        _, ref_hit = o.render_pixel(x, y)
        assert hit.node == int(ref_hit[0]), (x, y)


@pytest.mark.parametrize("name,size,over", [("lecture5.sdl", (200, 150), {}), ("chessboard.sdl", (240, 135), {}),
                                            ("../tests/scenes/nested.sdl", None, {}), ("../tests/scenes/quirks.sdl", None, {}),
                                            ("../tests/scenes/stereo_dof.sdl", None, {}), ("../tests/scenes/sky.sdl", None, {})])
def test_global_memory_scene_form_equals_constant_block_form(name, size, over, monkeypatch):
    """C2RT_FORCE_GLOBAL=1 routes a small scene through the MODE_BIG kernels: same frame as the constant-block form."""
    g, o = both(os.path.join(SC, name), size, **over)
    const, _, st_c = g.render(seed=3, count_rays=True)
    monkeypatch.setenv("C2RT_FORCE_GLOBAL", "1")   # read at scene-create time
    big = c2.HostScene(os.path.join(SC, name))
    if size:
        big.set_frame_size(*size)
    big.override(**over)
    glob, _, st_g = big.render(seed=3, count_rays=True)
    ref, ost = o.render(seed=3)
    assert_parity(glob, ref, what="global-memory form " + name)
    assert (st_g.primary_rays, st_g.shadow_rays) == (st_c.primary_rays, st_c.shadow_rays) == (ost.primary_rays, ost.shadow_rays)
    assert np.abs(glob - const).max() < 1e-5


def test_capacity_limits_are_errors(tmp_path):
    nodes = "".join('Node "n%d" { geometry "s"; shader "a"; translate %d 0 0 }; ' % (i, 3 * i) for i in range(4097))
    p = tmp_path / "many.sdl"
    p.write_text('Scene { Camera { pos 0 0 -50; fov 60 }\n Geometries { Sphere "s" { R 1 } }\n Shaders { Lambert "a" { color 1 1 1 } }\n Nodes { %s } }' % nodes)
    g = c2.HostScene(p)
    with pytest.raises(c2.C2rtError, match="too many nodes"):
        g.render()
    lights = "".join('PointLight "l%d" { pos %d 50 0; color 1 1 1; power 100 }; ' % (i, i) for i in range(9))
    p.write_text('Scene { Camera { pos 0 0 -50; fov 60 }\n Lights { %s } }' % lights)
    with pytest.raises(c2.C2rtError, match="too many lights"):
        c2.HostScene(p).render()


def test_many_scenes_alive_and_scene_switching():
    paths = ["lecture4.sdl", "lecture5.sdl", "lecture4-proc-texture.sdl"]
    gs = [c2.HostScene(os.path.join(SC, p)) for p in paths]
    refs = []
    for p, g in zip(paths, gs):
        g.set_frame_size(96, 64)
        o = OracleScene(os.path.join(SC, p))
        o.set_frame_size(96, 64)
        refs.append(o.render()[0])
    for _ in range(2):
        for g, ref in zip(gs, refs):
            assert_parity(g.render()[0], ref)


def test_argb_only_delivery():
    """c2rt_render with rgb == NULL: the interactive host's frame (only the packed plane SDL2Gui.draw blits comes back)."""
    g = c2.HostScene(os.path.join(SC, "lecture5.sdl"))
    g.set_frame_size(333, 217)
    rgb, argb, _ = g.render(argb=True)
    none, only, st = g.render(argb_only=True)
    assert none is None and st.launches >= 1
    np.testing.assert_array_equal(only, argb)
    np.testing.assert_array_equal(only, pack_rgb32(rgb))
    cam, stt = g.frame_blocks()
    assert api.lib.c2rt_render(g.device_scene(), C.byref(cam), C.byref(stt), None, None, None) == -1   # both planes NULL


def test_cancel_stops_a_frame_in_flight():
    """c2rt_cancel from another thread (the reference polls its stop flag between passes: renderer.d:93-97,129,147,180): tiles that
    have not started are skipped, c2rt_render reports C2RT_CANCELLED, and the next frame is complete again."""
    import threading
    import time
    g = c2.HostScene(os.path.join(SC, "zaphod.sdl"))      # DOF, 125 rays per pixel: ~16 ms of kernel at 4K
    g.set_frame_size(3840, 2160)
    buf = np.empty((2160, 3840, 3), np.float32)
    _, _, full = g.render(seed=1, out=buf)
    assert not g.cancelled
    reference = buf.copy()
    api.cancel()                                           # no frame in progress: cancels nothing
    _, _, st = g.render(seed=1, out=buf)
    assert not g.cancelled
    np.testing.assert_array_equal(buf, reference)
    started = threading.Event()
    res = {}

    def worker():
        started.set()
        res["st"] = g.render(seed=1, out=buf)[2]

    t = threading.Thread(target=worker)
    t.start()
    started.wait()
    time.sleep(0.004)
    api.cancel()
    t.join()
    assert g.cancelled
    assert res["st"].kernel_ms < 0.85 * full.kernel_ms, (res["st"].kernel_ms, full.kernel_ms)
    _, _, st = g.render(seed=1, out=buf)                   # the flag does not outlive the cancelled frame
    assert not g.cancelled
    np.testing.assert_array_equal(buf, reference)


def test_headless_end_to_end_and_orbit(tmp_path):
    """chess2rt_headless: the image files hold the frame the library renders (BMP through saveBmp's reference layout, PFM floats),
    and --orbit runs the camera-move loop with ARGB-only delivery."""
    import subprocess
    exe = os.path.join(ROOT, "chess2rt_b200", "chess2rt_headless")
    bmp, pfm = tmp_path / "o.bmp", tmp_path / "o.pfm"
    r = subprocess.run([exe, "--headless", "--file", os.path.join(SC, "lecture5.sdl"), "--width", "200", "--height", "120", "--out", str(bmp),
                        "--pfm", str(pfm), "--orbit", "6"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert "orbit: 6 frames of 200x120, ARGB-only delivery" in r.stdout
    g = c2.HostScene(os.path.join(SC, "lecture5.sdl"))
    g.set_frame_size(200, 120)
    rgb, argb, _ = g.render(argb=True)
    assert bmp.read_bytes() == api.save_bmp(argb)
    raw = pfm.read_bytes()
    head = b"PF\n200 120\n-1.0\n"
    assert raw.startswith(head)
    got = np.frombuffer(raw[len(head):], np.float32).reshape(120, 200, 3)[::-1]
    np.testing.assert_array_equal(got, rgb)


def test_fma_peak_microbenchmarks_are_sane():
    tf32, mhz = c2.measure_fma_peak(False)
    tf64, _ = c2.measure_fma_peak(True)
    assert 40 < tf32 < 90 and 15 < tf64 < 45 and 1000 < mhz < 2100
