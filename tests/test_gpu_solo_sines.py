"""Procedure2's u sines shared by frequency (render_kernel.cu texture_uv, scene_dev.h MODE_UPAT): a one-plane Procedure2 scene whose
u frequencies repeat gets a render_solo_kernel<..., ROWS_YZ> whose straight-line tap takes one sine per distinct frequency.  The
host judges "the same frequency" by the bits of the double the kernel multiplies u by (c2rt_api.cu proc2_u_pattern).  Every frame
must be BIT-identical to the general kernel (C2RT_NO_SOLO_FAST=1), the ARGB plane and the ray counts included, and each scene
checks the pattern its kernel is chosen by (c2rt_selftest_scene_class, no GPU needed)."""
import ctypes as C
import math
import os

import numpy as np
import pytest

import chess2rt_b200 as c2
from chess2rt_b200 import api
from test_gpu_solo_rows import assert_same_as_general, camera_rows
from test_gpu_solo_tiles import fast_and_general, render_device_bands

MODE_SOLO, MODE_UPAT_SHIFT = 32, 10
UPAT_DISTINCT, UPAT_01, UPAT_02, UPAT_12, UPAT_ALL = range(5)


def freq_d(f):
    """The double the kernel multiplies u by: the frequency in 2^-32 revolutions (c2rt_api.cu validate_and_build)."""
    return f / 6.283185307179586476925 * 4294967296.0


def next_distinct(f):
    """The first double above f whose kernel frequency has other bits than f's."""
    g = np.nextafter(f, math.inf)
    while freq_d(g) == freq_d(f):
        g = np.nextafter(g, math.inf)
    return float(g)


LAST_BIT = next_distinct(0.01)
# u frequencies of each pattern (lecture4-proc-texture.sdl has 0.01 0.25 0.01)
PATTERNS = {
    "distinct": ((0.01, 0.25, 0.03), UPAT_DISTINCT),
    "0=1": ((0.01, 0.01, 0.25), UPAT_01),
    "0=2": ((0.01, 0.25, 0.01), UPAT_02),
    "1=2": ((0.25, 0.01, 0.01), UPAT_12),
    "all": ((0.01, 0.01, 0.01), UPAT_ALL),
    "last_bit": ((0.01, 0.25, LAST_BIT), UPAT_DISTINCT),
}
SHADERS = {
    "lambert": 'Lambert "s" { texture "t" }',
    "phong": 'Phong "s" { color 0.9 0.8 0.7; exponent 40; strength 1; texture "t" }',
}


def write_scene(tmp_path, freq_u, shader="lambert", w=320, h=187):
    fu = " ".join(repr(float(f)) for f in freq_u)
    text = f"""Scene {{
  Name "sines"
  GlobalSettings {{ frameWidth {w}; frameHeight {h}; ambientLightColor 0.0 0.0 0.0; AAEnabled true; prepassEnabled false }}
  Camera {{ pos 0.0 165.0 0.0; yaw 0.0; pitch -30.0; roll 0.0; fov 90.0 }}
  Lights {{ PointLight "l1" {{ pos -30.0 100.0 250.0; color 1.0 1.0 1.0; power 50000 }} }}
  Geometries {{ Plane "floor" {{ y 2 }} }}
  Textures {{ Procedure2 "t" {{
      freqU {fu}
      freqV 0.01 0.25 0.01
      colorU {{ color 0.7 0.1 0.2; color 0.3 0.4 0.9; color 0.5 0.8 0.1 }}
      colorV {{ color 0.5 0.8 0.1; color 0.7 0.1 0.2; color 0.3 0.4 0.9 }}
  }} }}
  Shaders {{ {SHADERS[shader]} }}
  Nodes {{ Node "floor" {{ geometry "floor"; shader "s" }} }}
}}
"""
    path = tmp_path / f"sines_{abs(hash((fu, shader))) % 10**8}.sdl"
    path.write_text(text)
    return c2.HostScene(str(path))


def scene_class(g):
    return api.lib.c2rt_selftest_scene_class(C.cast(g.desc(), C.c_void_p))


def u_pattern(g):
    mode = scene_class(g)
    assert mode >= 0 and mode & MODE_SOLO, mode
    return mode >> MODE_UPAT_SHIFT


@pytest.mark.parametrize("name", list(PATTERNS) + ["zero_signs", "zero_signs_12"])
def test_host_derives_the_u_pattern_from_the_bits(name, tmp_path, monkeypatch):
    """No GPU: the pattern of each u-frequency set; 0.0 and -0.0 are different doubles, so they share no sine."""
    monkeypatch.delenv("C2RT_NO_SOLO", raising=False)
    freq_u, expect = {"zero_signs": ((0.0, -0.0, 0.0), UPAT_02), "zero_signs_12": ((-0.0, 0.0, 0.0), UPAT_12)}.get(name) or PATTERNS[name]
    g = write_scene(tmp_path, freq_u)
    assert u_pattern(g) == expect
    assert freq_d(LAST_BIT) != freq_d(0.01)
    monkeypatch.setenv("C2RT_NO_SOLO", "1")   # the general plane-only class: no one-plane kernel, no pattern
    assert scene_class(g) >> MODE_UPAT_SHIFT == 0 and not scene_class(g) & MODE_SOLO


@pytest.fixture(scope="module")
def ctx():
    c2.init(1, [0])
    yield
    c2.shutdown()


@pytest.mark.gpu
@pytest.mark.parametrize("shader", list(SHADERS))
@pytest.mark.parametrize("name", list(PATTERNS))
def test_u_patterns_equal_the_general_kernel(name, shader, ctx, tmp_path, monkeypatch):
    """Yaw 0 and roll 0 (the z table) at pitches with the horizon in the frame, ragged sizes, the launch's strips and forced ones."""
    freq_u, expect = PATTERNS[name]
    g = write_scene(tmp_path, freq_u, shader)
    assert u_pattern(g) == expect
    horizon, lit = 0, 0.0
    for d_pitch, strip in ((0.0, None), (24.0, 3), (30.0, None), (10.0, 2), (-20.0, 5)):
        if strip is None:
            monkeypatch.delenv("C2RT_SOLO_STRIP", raising=False)
        else:
            monkeypatch.setenv("C2RT_SOLO_STRIP", str(strip))
        g.camera_rotate(0.0, 0.0, d_pitch)
        for w, h in ((320, 187), (333, 61), (66, 9)):
            g.set_frame_size(w, h)
            cam, _ = g.frame_blocks(seed=5)
            assert cam.up_right[1] == cam.up_left[1] and cam.up_right[2] == cam.up_left[2], "du.y == du.z == 0: the z table"
            dy, _ = camera_rows(g)
            below = np.signbit(dy).all(axis=1)
            horizon += bool(below.any() and not below.all())
            rgb = assert_same_as_general(g, monkeypatch, f"{name} {shader} pitch {d_pitch} strip {strip} {w}x{h}")
            lit = max(lit, float(rgb.max()))
        g.camera_rotate(0.0, 0.0, -d_pitch)
    assert horizon > 0 and lit > 0.05, (horizon, lit)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["0=2", "all", "1=2"])
def test_aa_off_argb_only_and_row_bands(name, ctx, tmp_path, monkeypatch):
    freq_u, expect = PATTERNS[name]
    g = write_scene(tmp_path, freq_u)
    assert u_pattern(g) == expect
    monkeypatch.setenv("C2RT_SOLO_STRIP", "3")
    g.override(aa=0)
    for w, h in ((333, 187), (31, 9)):
        g.set_frame_size(w, h)
        (rgb, argb, st), (rgb_g, argb_g, st_g) = fast_and_general(monkeypatch, lambda: g.render(argb=True, seed=5, count_rays=True))
        np.testing.assert_array_equal(rgb, rgb_g, err_msg=f"aa off {w}x{h}")
        np.testing.assert_array_equal(argb, argb_g, err_msg=f"aa off {w}x{h}")
        assert (st.primary_rays, st.shadow_rays) == (st_g.primary_rays, st_g.shadow_rays) and st.primary_rays == w * h
    g.override(aa=1)
    monkeypatch.delenv("C2RT_SOLO_STRIP")
    g.set_frame_size(333, 187)
    (none, only, _), (_, only_g, _) = fast_and_general(monkeypatch, lambda: g.render(argb_only=True, seed=5))
    assert none is None
    np.testing.assert_array_equal(only, only_g)
    full, full_a, _ = g.render(argb=True, seed=5)
    np.testing.assert_array_equal(only, full_a)
    for compact in (0, 1):
        (rgb, argb), (rgb_g, argb_g) = fast_and_general(monkeypatch, lambda: render_device_bands(g, 3, 16, compact))
        np.testing.assert_array_equal(rgb, rgb_g)
        np.testing.assert_array_equal(argb, argb_g)
        np.testing.assert_array_equal(rgb, full)
        np.testing.assert_array_equal(argb, full_a)
