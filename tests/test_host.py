"""Host-side logic without a GPU: the C ABI library loads and exports every symbol of include/c2rt.h,
the reference-compatible loader + flattener produce the expected structure-of-arrays description,
load errors mirror the reference's exception behaviour, the render entry points fail LOUDLY (no CPU
fallback), band arithmetic, and the world_size-2 gather path over gloo."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import chess2rt_b200 as c2
from chess2rt_b200 import api, bands
from bmp_kats import KAT1, KAT1_PIXELS, KAT1_SIZE, KAT2, KAT2_PIXELS, KAT2_SIZE
from oracle_binding import OracleScene, oracle_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SC = os.path.join(ROOT, "scenes")
HAS_GPU = c2.device_count() > 0


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "c2rt.h")).read()
    declared = set(re.findall(r"\b(c2rt_[a-z0-9_]+)\s*\(", header))
    declared -= {"c2rt_status"}
    assert declared == set(api.C_ABI_SYMBOLS), declared ^ set(api.C_ABI_SYMBOLS)
    for name in declared:
        assert hasattr(api.lib, name), name
    assert api.lib.c2rt_abi_version() == 2
    # no torch / C++ types at the boundary: the exported names are unmangled C
    out = subprocess.run(["nm", "-D", "--defined-only", os.path.join(ROOT, "chess2rt_b200", "libc2rt.so")],
                         capture_output=True, text=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    assert declared <= exported


@pytest.mark.parametrize("workers,rounds", [(1, 3000), (7, 3000), (15, 1000)])
def test_device_pool_hands_every_frame_to_every_worker(workers, rounds):
    """The helper threads of the multi-device c2rt_render (one per extra device): no frame lost or run twice,
    across the spinning and the sleeping hand-off and a pool restart (no GPU involved)."""
    assert api.lib.c2rt_selftest_device_pool(workers, rounds) == workers * rounds
    assert api.lib.c2rt_selftest_device_pool(0, 1) < 0


def test_struct_layouts_match_header_sizes():
    # sizes the C compiler gives the ABI structs (x86-64 SysV): guards the ctypes mirrors
    assert C.sizeof(api.Camera) == 7 * 24 + 4 * 4 + 3 * 8
    assert C.sizeof(api.Settings) == 64
    assert C.sizeof(api.Band) == 16 + 8 + 4 + 4   # + done_flags pointer, frame_no, reserved
    assert C.sizeof(api.Stats) == 40
    assert C.sizeof(api.Hit) == 8 + 8 + 24 + 24 + 16
    s = c2.HostScene(os.path.join(SC, "lecture4.sdl"))
    assert s.desc().contents.struct_size == C.sizeof(api.SceneDesc)


def test_loader_and_flattener_lecture5():
    s = c2.HostScene(os.path.join(SC, "lecture5.sdl"))
    assert s.info() == {"nodes": 6, "geometries": 6, "shaders": 4, "textures": 2, "lights": 1, "aa": 1, "dof": 0,
                        "num_samples": 25}
    assert s.frame_size == (640, 480)
    d = s.desc().contents
    assert (d.n_nodes, d.n_geoms, d.n_shaders, d.n_textures, d.n_lights) == (6, 6, 4, 2, 1)
    gt = [d.geom_type[i] for i in range(6)]
    assert gt == [0, 1, 2, 1, 5, 1]  # plane, sphere, cube, sphere, CsgDiff, sphere
    assert (d.geom_left[4], d.geom_right[4]) == (2, 3)          # references became indices
    assert [d.node_geom[i] for i in range(6)] == [0, 1, 4, 5, 5, 5]  # the shared sphere "S" keeps ONE entry
    assert [d.node_shader[i] for i in range(6)] == [0, 1, 2, 3, 3, 3]
    np.testing.assert_array_equal([d.node_offset[3 * 3 + k] for k in range(3)], [100, 15, 256])
    assert [d.node_transform[9 * 3 + k] for k in range(9)] == [1, 0, 0, 0, 1, 0, 0, 0, 1]
    assert (d.tex_width[0], d.tex_height[0], d.tex_width[1], d.tex_height[1]) == (256, 256, 800, 400)
    assert d.tex_texel_offset[1] == 256 * 256 and d.n_texels == 256 * 256 + 800 * 400
    assert abs(d.tex_params[0] - float(np.float32(0.005))) == 0  # float scaling widened exactly
    assert d.shader_exponent[2] == 60 and d.shader_exponent[3] == 80 and d.shader_strength[2] == 1
    assert np.isnan(d.geom_params[1])  # Plane.limit stays NaN -> unbounded
    # texels handed to the backend are bit-identical to the oracle's post-gamma Image!Color
    o = OracleScene(os.path.join(SC, "lecture5.sdl"))
    tex0 = o.texture_texels(0)
    got = np.ctypeslib.as_array(d.texels, shape=(d.n_texels * 3,))[: 256 * 256 * 3].reshape(256, 256, 3)
    np.testing.assert_array_equal(got, tex0)


def test_cubemap_environment_extension_is_loaded_and_flattened(tmp_path):
    """Environment { folder ... } (EXTENSION; the reference's Environment reads no keys, environment.d:12-14): six faces loaded
    with the BitmapTexture gamma rule and appended to the flat texel array; scenes without it keep C2RT_ENV_BLACK."""
    plain = c2.HostScene(os.path.join(SC, "lecture5.sdl"))
    d = plain.desc().contents
    assert d.env_type == 0 and d.n_texels == 256 * 256 + 800 * 400
    s = c2.HostScene(os.path.join(ROOT, "tests", "scenes", "sky.sdl"))
    d = s.desc().contents
    assert d.env_type == 1 and d.n_textures == 1 and d.n_texels == 6 * 128 * 128
    assert list(d.env_face_width) == [128] * 6 and list(d.env_face_height) == [128] * 6
    assert list(d.env_face_texel_offset) == [k * 128 * 128 for k in range(6)]
    # the texels handed over equal the oracle's post-gamma faces (posy, top-left texel, through its lookup at the face corner)
    o = OracleScene(os.path.join(ROOT, "tests", "scenes", "sky.sdl"))
    got = np.ctypeslib.as_array(d.texels, shape=(d.n_texels * 3,)).reshape(6, 128, 128, 3)
    np.testing.assert_array_equal(got[2, 0, 0], o.environment((-1, 1, -1))[1])      # posy: (sx, sy) = (vx, vz) = (-1, -1)
    np.testing.assert_array_equal(got[5, 127, 127], o.environment((-1, -1, -1))[1])  # negz: (-vx, -vy) = (1, 1) -> last texel
    p = tmp_path / "nofaces.sdl"
    p.write_text('Scene { Environment { folder "nowhere" } }')
    with pytest.raises(c2.C2rtError):
        c2.HostScene(p)


def test_save_bmp_is_the_reference_layout():
    """imageio/bmp.d:195-237 by hand for a 3x2 image: 14-byte file header (fileSize = 54 + 3 W H, offset 54), BITMAPINFOHEADER
    (40, W, H, 1 plane, 24 bpp, BI_RGB, size = fileSize - 54, 72 dpi = lrint(7200 / 2.54) = 2835 px/m twice, 0, 0), then the rows
    from the BOTTOM one up, each pixel the low three little-endian bytes of Color.toRGB32 (b, g, r) — and no row padding
    (3 * 3 = 9 bytes per row), which makes the reference's own loader (bmp.d:136-188, padded rows) misread such a file."""
    import struct
    argb = np.array([[0x00112233, 0x00445566, 0x00778899], [0x00AABBCC, 0x00DDEEFF, 0x00010203]], np.uint32)
    got = api.save_bmp(argb)
    head = struct.pack("<2sIHHI", b"BM", 54 + 18, 0, 0, 54) + struct.pack("<IiiHHIIiiII", 40, 3, 2, 1, 24, 0, 18, 2835, 2835, 0, 0)
    rows = bytes([0xCC, 0xBB, 0xAA, 0xFF, 0xEE, 0xDD, 0x03, 0x02, 0x01]) + bytes([0x33, 0x22, 0x11, 0x66, 0x55, 0x44, 0x99, 0x88, 0x77])
    assert got == head + rows
    # --pad-rows: the valid file; PIL and the host's own decoder read the pixels back
    from io import BytesIO
    from PIL import Image
    padded = api.save_bmp(argb, pad_rows=True)
    assert len(padded) == 54 + 2 * 12
    img = np.asarray(Image.open(BytesIO(padded)).convert("RGB")).astype(np.uint32)
    np.testing.assert_array_equal((img[..., 0] << 16) | (img[..., 1] << 8) | img[..., 2], argb)
    w, h = C.c_uint32(), C.c_uint32()
    out = np.zeros(6, np.uint32)
    blob = np.frombuffer(padded, np.uint8)
    assert api.host_lib.c2rt_host_decode_bmp(blob.ctypes.data, blob.size, C.byref(w), C.byref(h), out.ctypes.data, 6) == 0
    np.testing.assert_array_equal(out.reshape(2, 3), argb)
    # widths with 3 W % 4 == 0 need no padding: both forms coincide
    a4 = np.arange(8, dtype=np.uint32).reshape(2, 4) * 0x010203
    assert api.save_bmp(a4) == api.save_bmp(a4, pad_rows=True)


def test_headless_command_line(tmp_path):
    """chess2rt_headless (host/main.cpp, the C++ twin of integration/d/source/app_headless.d): usage errors exit 2, load errors exit 1 with
    the reference's message, and without a GPU a render fails loudly (no CPU fallback) instead of writing an image."""
    exe = os.path.join(ROOT, "chess2rt_b200", "chess2rt_headless")
    run = lambda *a: subprocess.run([exe, *a], capture_output=True, text=True, timeout=300)
    r = run()
    assert r.returncode == 2 and "usage:" in r.stderr
    assert run("--file").returncode == 2 and run("--bogus", "1").returncode == 2
    assert run("--file", os.path.join(SC, "lecture4.sdl"), "--gpus", "0").returncode == 2
    r = run("--file", str(tmp_path / "missing.sdl"))
    assert r.returncode == 1 and "Scene file not found" in r.stderr
    out = tmp_path / "x.bmp"
    r = run("--headless", "--file=" + os.path.join(SC, "lecture4.sdl"), "--width", "64", "--height", "48", "--out", str(out))
    if HAS_GPU:
        assert r.returncode == 0 and out.exists() and out.stat().st_size == 54 + 64 * 48 * 3
    else:
        assert r.returncode == 1 and "CUDA" in r.stderr and not out.exists()


def test_settings_block_carries_the_gi_fields(tmp_path):
    """GlobalSettings -> c2rt_settings (flatten.cpp flattenSettings): GIEnabled / pathsPerPixel / bucketSize reach the ABI."""
    from test_oracle_kat import GI_SCENE
    p = tmp_path / "gi.sdl"
    p.write_text(GI_SCENE.format(paths=6, cam="", ball_shader="Lambert"))
    _, st = c2.HostScene(str(p)).frame_blocks(seed=9)
    assert (st.gi_enabled, st.paths_per_pixel, st.max_trace_depth, st.bucket_size, st.rng_seed) == (1, 6, 3, 48, 9)
    assert (st.frame_width, st.frame_height, st.aa_enabled) == (96, 64, 1)
    _, st = c2.HostScene(os.path.join(SC, "lecture4.sdl")).frame_blocks()
    assert (st.gi_enabled, st.paths_per_pixel) == (0, 40)   # global_settings.d:8-35 defaults


def test_loader_json_equals_sdl_and_quirks():
    a = c2.HostScene(os.path.join(SC, "lecture4.sdl"))
    b = c2.HostScene(os.path.join(SC, "lecture4.json"))
    ia, ib = a.info(), b.info()
    assert ia["aa"] == 1 and ib["aa"] == 0
    ia.pop("aa"), ib.pop("aa")
    assert ia == ib
    da, db = a.desc().contents, b.desc().contents
    assert [da.tex_colors[i] for i in range(6)] == [db.tex_colors[i] for i in range(6)]
    # Node "rotate" is applied as a second scale (node.d:89-90)
    q = c2.HostScene(os.path.join(ROOT, "tests", "scenes", "quirks.sdl"))
    d = q.desc().contents
    m = [d.node_transform[9 * 7 + k] for k in range(9)]  # "globe": scale 1.2 0.9 1.2 then rotate 1 1.1 1
    np.testing.assert_allclose(m, [1.2, 0, 0, 0, 0.9 * 1.1, 0, 0, 0, 1.2], rtol=1e-15)
    inv = [d.node_inverse[9 * 7 + k] for k in range(9)]
    np.testing.assert_allclose(inv[4], 1 / (0.9 * 1.1), rtol=1e-15)
    # camera blocks agree with the oracle's Camera.beginFrame
    cam, st = q.frame_blocks()
    o = OracleScene(os.path.join(ROOT, "tests", "scenes", "quirks.sdl"))
    v = o.camera_vectors()
    got = np.array([list(cam.pos), list(cam.up_left), list(cam.up_right), list(cam.down_left), list(cam.right_dir),
                    list(cam.up_dir), list(cam.front_dir)])
    np.testing.assert_array_equal(got, v)
    assert (st.frame_width, st.frame_height, st.aa_enabled, st.prepass_enabled) == (320, 200, 1, 0)


def test_load_errors_mirror_reference(tmp_path):
    with pytest.raises(c2.C2rtError, match="Scene file not found"):   # scene_loader.d:29-32
        c2.HostScene(tmp_path / "missing.sdl")
    p = tmp_path / "x.txt"
    p.write_text("Scene {}")
    with pytest.raises(c2.C2rtError, match="unknown file type"):       # scene_loader.d:56-58
        c2.HostScene(p)
    p = tmp_path / "bad.sdl"
    p.write_text("Scene {\n Geometries {\n  Torus \"t\" { R 1 }\n }\n}\n")
    with pytest.raises(c2.C2rtError, match="Unknown object type"):     # scene_loader.d:189-191
        c2.HostScene(p)
    p = tmp_path / "dup.sdl"
    p.write_text("Scene {\n Geometries {\n  Sphere \"a\" { R 1 }\n  Sphere \"a\" { R 2 }\n }\n}\n")
    with pytest.raises(c2.C2rtError, match="duplicate name"):          # scene_loader.d:198
        c2.HostScene(p)
    p = tmp_path / "brace.sdl"
    p.write_text("Scene {\n Geometries {\n")
    with pytest.raises(c2.C2rtError, match="Invalid SDL"):             # scene_loader.d:37-40
        c2.HostScene(p)
    p = tmp_path / "bad.json"
    p.write_text("{ \"Camera\": ")
    with pytest.raises(c2.C2rtError, match="Invalid JSON"):            # scene_loader.d:33-36
        c2.HostScene(p)


@pytest.mark.parametrize("blob,size,pixels", [(KAT1, KAT1_SIZE, KAT1_PIXELS), (KAT2, KAT2_SIZE, KAT2_PIXELS)])
def test_host_bmp_decoder_reference_kats(blob, size, pixels):
    w, h = C.c_uint32(), C.c_uint32()
    out = np.zeros(16, np.uint32)
    buf = np.frombuffer(blob, np.uint8)
    assert api.host_lib.c2rt_host_decode_bmp(buf.ctypes.data, len(blob), C.byref(w), C.byref(h), out.ctypes.data, out.size) == 0
    assert (w.value, h.value) == size
    assert [int(v) for v in out[: len(pixels)]] == [p & 0xFFFFFF for p in pixels]  # Color has no alpha


def test_validation_errors_come_before_any_device_use(tmp_path):
    # CSG nesting deeper than 3 levels is rejected with C2RT_ERR_UNSUPPORTED by the scene validator (no GPU needed)
    p = tmp_path / "nested.sdl"
    p.write_text("""Scene {
 Geometries {
  Sphere "a" { R 1 }
  Cube "b" { side 1 }
  CsgUnion "u1" { left "a"; right "b" }
  CsgDiff "u2" { left "u1"; right "a" }
  CsgInter "u3" { left "u2"; right "b" }
  CsgUnion "u4" { left "a"; right "u3" }
 }
 Shaders { Lambert "s" { color 1 1 1 } }
 Nodes { Node "n" { geometry "u4"; shader "s" } }
}
""")
    s = c2.HostScene(p)
    d = s.desc()
    handle = C.c_void_p()
    rc = api.lib.c2rt_scene_create(d, C.byref(handle))
    assert rc == -2 and b"nesting deeper" in api.lib.c2rt_last_error()
    # ABI mismatch
    bad = api.SceneDesc()
    assert api.lib.c2rt_scene_create(C.byref(bad), C.byref(handle)) == -1
    assert api.lib.c2rt_scene_create(None, C.byref(handle)) == -1


@pytest.mark.skipif(HAS_GPU, reason="checks the no-GPU behaviour")
def test_render_fails_loudly_without_a_gpu():
    s = c2.HostScene(os.path.join(SC, "lecture4.sdl"))
    with pytest.raises(c2.C2rtError, match="no CPU fallback"):
        s.render()
    with pytest.raises(c2.C2rtError):
        c2.init(1)


def test_pinned_rng_is_shared_between_oracle_and_library():
    lib = oracle_lib()
    rng = np.random.default_rng(1)
    for _ in range(200):
        seed = int(rng.integers(0, 2**63))
        px, py, tap, smp, draw = [int(v) for v in rng.integers(0, 8000, 5)]
        v = c2.rng_u31(seed, px, py, tap, smp, draw)
        assert v == lib.orc_rng_u31(seed, px, py, tap, smp, draw)
        assert 0 <= v < 2**31
    vals = np.array([c2.rng_u31(9, x, y, 0, 0, 0) for x in range(64) for y in range(64)]) / 2147483647.0
    assert abs(vals.mean() - 0.5) < 0.02 and abs(vals.var() - 1 / 12) < 0.01


def test_srgb_table_of_the_library_equals_the_oracle_table():
    from oracle_binding import srgb_lut
    np.testing.assert_array_equal(c2.srgb_table(), srgb_lut())


@pytest.mark.parametrize("h,n,b", [(1080, 8, 8), (1080, 3, 16), (430, 4, 8), (7, 2, 8), (4320, 8, 8), (100, 1, 8)])
def test_band_arithmetic(h, n, b):
    total = 0
    seen = np.zeros(h, int)
    for r in range(n):
        rows = bands.owned_rows(h, r, n, b)
        assert c2.band_rows_owned(h, r, n, b) == rows.size
        seen[rows] += 1
        total += rows.size
    assert total == h and np.all(seen == 1)
    assert bands.rows_padded(h, n, b) == max(bands.rows_owned(h, r, n, b) for r in range(n))
    g = np.zeros((n, bands.rows_padded(h, n, b), 3), np.int64)
    for r in range(n):
        rows = bands.owned_rows(h, r, n, b)
        g[r, : rows.size, 0] = rows
    np.testing.assert_array_equal(bands.scatter_rows(g, h, n, b)[:, 0], np.arange(h))


def test_two_rank_band_gather_over_gloo(tmp_path):
    """world_size 2 on CPU (gloo): each rank produces its interleaved bands (with the oracle standing in
    for the kernel), rank 0 gathers + scatters; the assembled frame equals the single-rank frame."""
    script = os.path.join(ROOT, "tests", "_gloo_band_worker.py")
    out = tmp_path / "ok.txt"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", script, str(out)]
    env = dict(os.environ, OMP_NUM_THREADS="1")
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert out.read_text().strip() == "ok"


def test_json_and_sdl_forms_of_every_object_type_agree(tmp_path):
    """The same scene written in both formats (scene_loader.d:243-403): JSON objects carry "type"/"name" members,
    Vector/Color are number arrays, arrays of Color are arrays of arrays, scalar arrays plain arrays."""
    sdl = '''Scene {
  Name "both"
  GlobalSettings { frameWidth 48; frameHeight 32; ambientLightColor 0.1 0.2 0.3; AAEnabled false; bucketSize 16 }
  Camera { pos 1 60 -90; yaw 3; pitch -25; roll 1; fov 70; focalPlaneDist 80; fNumber 4; numSamples 3; stereoSeparation 0 }
  Lights { PointLight "l" { pos -50 200 -40; color 1 0.9 0.8; power 30000 } }
  Geometries {
    Plane "f" { y 1 }
    Sphere "s" { center 0 20 0; R 18 }
    Cube { name "c"; center 2 20 1; side 30 }
    CsgDiff "d" { left "c"; right "s" }
  }
  Textures {
    Checker "chk" { color1 0.1 0.1 0.1; color2 0.9 0.8 0.7; size 6 }
    Procedure2 "p" { freqU 0.1 0.2 0.3; freqV 0.3 0.2 0.1
      colorU { color 0.1 0.2 0.3; color 0.3 0.2 0.1; color 0.2 0.2 0.2 }
      colorV { color 0.3 0.1 0.1; color 0.1 0.3 0.1; color 0.1 0.1 0.3 } }
    BitmapTexture "b" { file "%(sc)s/floor.bmp"; scaling 0.01; assumedGamma 2.2 }
  }
  Shaders {
    Lambert "a" { texture "chk" }
    Phong "b" { color 0.7 0.3 0.2; exponent 33; strength 0.5; texture "p" }
    Lambert "c" { texture "b" }
  }
  Nodes {
    Node "n0" { geometry "f"; shader "c" }
    Node "n1" { geometry "d"; shader "b"; scale 1 1.2 1; rotate 1.1 1 0.9; translate -20 5 10 }
    Node "n2" { geometry "s"; shader "a"; translate 40 0 30 }
  }
}''' % {"sc": SC}
    js = '''{
  "Name": "both",
  "GlobalSettings": {"type": "GlobalSettings", "frameWidth": 48, "frameHeight": 32, "ambientLightColor": [0.1, 0.2, 0.3], "AAEnabled": false, "bucketSize": 16},
  "Camera": {"type": "Camera", "pos": [1, 60, -90], "yaw": 3, "pitch": -25, "roll": 1, "fov": 70, "focalPlaneDist": 80, "fNumber": 4, "numSamples": 3, "stereoSeparation": 0},
  "Lights": [{"type": "PointLight", "name": "l", "pos": [-50, 200, -40], "color": [1, 0.9, 0.8], "power": 30000}],
  "Geometries": [
    {"type": "Plane", "name": "f", "y": 1},
    {"type": "Sphere", "name": "s", "center": [0, 20, 0], "R": 18},
    {"type": "Cube", "name": "c", "center": [2, 20, 1], "side": 30},
    {"type": "CsgDiff", "name": "d", "left": "c", "right": "s"}],
  "Textures": [
    {"type": "Checker", "name": "chk", "color1": [0.1, 0.1, 0.1], "color2": [0.9, 0.8, 0.7], "size": 6},
    {"type": "Procedure2", "name": "p", "freqU": [0.1, 0.2, 0.3], "freqV": [0.3, 0.2, 0.1],
     "colorU": [[0.1, 0.2, 0.3], [0.3, 0.2, 0.1], [0.2, 0.2, 0.2]], "colorV": [[0.3, 0.1, 0.1], [0.1, 0.3, 0.1], [0.1, 0.1, 0.3]]},
    {"type": "BitmapTexture", "name": "b", "file": "%(sc)s/floor.bmp", "scaling": 0.01, "assumedGamma": 2.2}],
  "Shaders": [
    {"type": "Lambert", "name": "a", "texture": "chk"},
    {"type": "Phong", "name": "b", "color": [0.7, 0.3, 0.2], "exponent": 33, "strength": 0.5, "texture": "p"},
    {"type": "Lambert", "name": "c", "texture": "b"}],
  "Nodes": [
    {"type": "Node", "name": "n0", "geometry": "f", "shader": "c"},
    {"type": "Node", "name": "n1", "geometry": "d", "shader": "b", "scale": [1, 1.2, 1], "rotate": [1.1, 1, 0.9], "translate": [-20, 5, 10]},
    {"type": "Node", "name": "n2", "geometry": "s", "shader": "a", "translate": [40, 0, 30]}]
}''' % {"sc": SC}
    ps, pj = tmp_path / "both.sdl", tmp_path / "both.json"
    ps.write_text(sdl)
    pj.write_text(js)
    # oracle: identical images
    a, b = OracleScene(ps), OracleScene(pj)
    ia, sa = a.render(threads=2)
    ib, sb = b.render(threads=2)
    np.testing.assert_array_equal(ia, ib)
    assert (sa.primary_rays, sa.shadow_rays) == (sb.primary_rays, sb.shadow_rays)
    # host loader + flattener: identical flat descriptions
    ha, hb = c2.HostScene(ps), c2.HostScene(pj)
    assert ha.info() == hb.info()
    da, db = ha.desc().contents, hb.desc().contents
    for name, n in [("node_transform", 27), ("node_inverse", 27), ("node_offset", 9), ("geom_params", 16), ("tex_params", 18),
                    ("shader_exponent", 3), ("light_pos", 3)]:
        va = np.array([getattr(da, name)[i] for i in range(n)])
        vb = np.array([getattr(db, name)[i] for i in range(n)])
        np.testing.assert_array_equal(va, vb, err_msg=name)   # NaN == NaN here (Plane.limit)
    for name, n in [("node_geom", 3), ("node_shader", 3), ("geom_type", 4), ("geom_left", 4), ("geom_right", 4), ("shader_type", 3),
                    ("shader_texture", 3), ("tex_type", 3)]:
        assert [getattr(da, name)[i] for i in range(n)] == [getattr(db, name)[i] for i in range(n)], name
    assert [da.tex_colors[i] for i in range(54)] == [db.tex_colors[i] for i in range(54)]
    ca, _ = ha.frame_blocks()
    cb, _ = hb.frame_blocks()
    assert bytes(ca) == bytes(cb)


# ---------------------------------------------------------------- the loader against an independent reader
SDL_FILES = ["scenes/lecture4.sdl", "scenes/lecture4-proc-texture.sdl", "scenes/lecture5.sdl", "scenes/zaphod.sdl",
             "scenes/chessboard.sdl", "tests/scenes/quirks.sdl", "tests/scenes/nested.sdl", "tests/scenes/sky.sdl"]
GEOM_TYPES = {"Plane": 0, "Sphere": 1, "Cube": 2, "CsgUnion": 3, "CsgInter": 4, "CsgDiff": 5}


def _vec(v):
    return list(v) if isinstance(v, (list, tuple)) else [v]


@pytest.mark.parametrize("path", SDL_FILES)
def test_loader_agrees_with_an_independent_sdl_reader(path):
    """host/scene_text.hpp parses the scene text for the host loader AND for the oracle, so a parse bug would be common-mode.
    tests/sdl_reader.py is a second, independent reader (Python, no shared code): every value it finds in the file must be the
    value the loader + flattener hand to the backend (indices for names, offsets / diagonal matrices for translate / scale)."""
    import sdl_reader as R
    scene = R.parse(open(os.path.join(ROOT, path)).read())[0]
    assert scene[0] == "Scene"
    host = c2.HostScene(os.path.join(ROOT, path))
    d = host.desc().contents
    cam, st = host.frame_blocks()
    sect = lambda n: (R.child(scene, n) or (n, [], []))[2]
    geoms, shaders, textures, lights, nodes = sect("Geometries"), sect("Shaders"), sect("Textures"), sect("Lights"), sect("Nodes")
    assert (d.n_geoms, d.n_shaders, d.n_textures, d.n_lights, d.n_nodes) == (len(geoms), len(shaders), len(textures), len(lights), len(nodes))
    gname = {R.obj_name(g): i for i, g in enumerate(geoms)}
    sname = {R.obj_name(s): i for i, s in enumerate(shaders)}
    tname = {R.obj_name(t): i for i, t in enumerate(textures)}
    for i, g in enumerate(geoms):
        assert d.geom_type[i] == GEOM_TYPES[g[0]], (path, i)
        p = [d.geom_params[4 * i + k] for k in range(4)]
        if g[0] == "Plane" and R.prop(g, "y") is not None:
            assert p[0] == float(R.prop(g, "y"))
        if g[0] in ("Sphere", "Cube"):
            if R.prop(g, "center") is not None:
                assert p[:3] == [float(x) for x in R.prop(g, "center")]
            key = "R" if g[0] == "Sphere" else "side"
            if R.prop(g, key) is not None:
                assert p[3] == float(R.prop(g, key))
        if g[0].startswith("Csg"):
            assert (d.geom_left[i], d.geom_right[i]) == (gname[R.prop(g, "left")], gname[R.prop(g, "right")])
    for i, s in enumerate(shaders):
        assert d.shader_type[i] == {"Lambert": 0, "Phong": 1}[s[0]]
        if R.prop(s, "color") is not None:
            np.testing.assert_array_equal([d.shader_color[3 * i + k] for k in range(3)], np.float32(R.prop(s, "color")))
        assert d.shader_texture[i] == (tname[R.prop(s, "texture")] if R.prop(s, "texture") is not None else -1)
        if s[0] == "Phong" and R.prop(s, "exponent") is not None:
            assert d.shader_exponent[i] == float(R.prop(s, "exponent"))
    for i, l in enumerate(lights):
        if R.prop(l, "pos") is not None:
            assert [d.light_pos[3 * i + k] for k in range(3)] == [float(x) for x in R.prop(l, "pos")]
        if R.prop(l, "power") is not None:
            assert d.light_power[i] == np.float32(R.prop(l, "power"))
        if R.prop(l, "color") is not None:
            np.testing.assert_array_equal([d.light_color[3 * i + k] for k in range(3)], np.float32(R.prop(l, "color")))
    for i, n in enumerate(nodes):
        assert d.node_geom[i] == gname[R.prop(n, "geometry")] and d.node_shader[i] == sname[R.prop(n, "shader")]
        off = [float(x) for x in R.prop(n, "translate", [0, 0, 0])]
        assert [d.node_offset[3 * i + k] for k in range(3)] == off
        diag = np.ones(3)
        for key in ("scale", "rotate"):   # node.d:89-90: `rotate` is applied as a second scale
            if R.prop(n, key) is not None:
                diag = diag * np.array([float(x) for x in R.prop(n, key)])
        M = np.array([d.node_transform[9 * i + k] for k in range(9)]).reshape(3, 3)
        np.testing.assert_allclose(M, np.diag(diag), rtol=1e-15)
    c = R.child(scene, "Camera")
    if c is not None and R.prop(c, "pos") is not None:
        assert list(cam.pos) == [float(x) for x in R.prop(c, "pos")]
    if c is not None and R.prop(c, "dof") is not None:
        assert bool(cam.dof) == R.prop(c, "dof")
    gs = R.child(scene, "GlobalSettings")
    if gs is not None:
        assert (st.frame_width, st.frame_height) == (R.prop(gs, "frameWidth", 640), R.prop(gs, "frameHeight", 480))
        if R.prop(gs, "ambientLightColor") is not None:
            np.testing.assert_array_equal(list(st.ambient_light), np.float32(R.prop(gs, "ambientLightColor")))
        if R.prop(gs, "AAEnabled") is not None:
            assert bool(st.aa_enabled) == R.prop(gs, "AAEnabled")


def test_json_loader_agrees_with_python_json():
    import json as pyjson
    j = pyjson.load(open(os.path.join(SC, "lecture4.json")))
    host = c2.HostScene(os.path.join(SC, "lecture4.json"))
    d = host.desc().contents
    cam, st = host.frame_blocks()
    assert list(cam.pos) == [float(x) for x in j["Camera"]["pos"]]
    assert (st.frame_width, st.frame_height, bool(st.aa_enabled)) == (j["GlobalSettings"]["frameWidth"], j["GlobalSettings"]["frameHeight"], j["GlobalSettings"]["AAEnabled"])
    assert d.n_lights == len(j["Lights"]) and d.n_nodes == len(j["Nodes"]) and d.n_geoms == len(j["Geometries"])
    L = j["Lights"][0]
    assert [d.light_pos[k] for k in range(3)] == [float(x) for x in L["pos"]] and d.light_power[0] == np.float32(L["power"])


def test_bench_parity_check_passes_the_oracle_and_fails_a_wrong_frame(tmp_path):
    """bench.py's parity check alongside timing (SURVEY.md section 8(d)), exercised on the CPU: fed the oracle's own rows it
    passes with a zero report, fed a frame with one pixel off by 2e-3 it reports that pixel and does not pass; the row windows
    cover the frame and the diff image is written for whole-frame checks."""
    import bench
    from oracle_binding import OracleScene
    path, w, h = "scenes/lecture4.sdl", 96, 64
    o = OracleScene(os.path.join(ROOT, path))
    o.set_frame_size(w, h)
    ref, _ = o.render(threads=2, seed=bench.RNG_SEED)
    diff = tmp_path / "diff.pgm"
    rep = bench.oracle_parity(path, w, h, {}, lambda y0, y1: ref[y0:y1], rows=None, diff_path=str(diff))
    assert rep["pass"] and rep["max_abs"] == 0.0 and rep["n"] == w * h and rep["sample"] == "whole frame"
    assert diff.read_bytes().startswith(b"P5\n96 64\n255\n") and len(diff.read_bytes()) == len(b"P5\n96 64\n255\n") + w * h
    bad = ref.copy()
    bad[40, 10, 1] += 2e-3
    asked = []

    def rows(y0, y1):
        asked.append((y0, y1))
        return bad[y0:y1]
    rep = bench.oracle_parity(path, w, h, {}, rows, rows=64)
    assert asked == [(8 * i, 8 * i + 8) for i in range(8)]          # 64 rows = the whole 64-row frame in windows of 8
    assert not rep["pass"] and rep["px_over_1e-3"] == 1 and abs(rep["max_abs"] - 2e-3) < 1e-6
    rep = bench.oracle_parity(path, w, h, {}, lambda y0, y1: bad[y0:y1], rows=16)   # two windows, rows 0-7 and 32-39: the bad pixel is outside
    assert rep["pass"] and rep["n"] == 16 * w


def test_bench_dump_frame_keeps_whole_frames_and_samples_rows_of_large_ones(tmp_path, monkeypatch):
    """bench.py --dump-outputs: a frame within the size limit is written whole; a larger one keeps every k-th row, the rows listed
    beside it, and the files stay within the limit."""
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    frame = np.random.default_rng(0).random((100, 2000, 3), dtype=np.float32)   # 2.4 MB
    bench.dump_frame(str(tmp_path / "small"), frame[:10])
    assert sorted(os.listdir(tmp_path / "small")) == ["frame.npy"]
    np.testing.assert_array_equal(np.load(tmp_path / "small" / "frame.npy"), frame[:10])
    bench.dump_frame(str(tmp_path / "big"), frame)
    rows = np.load(tmp_path / "big" / "frame_rows.npy")
    assert rows.dtype == np.float64 and rows[0] == 0 and len(set(np.diff(rows))) == 1
    np.testing.assert_array_equal(np.load(tmp_path / "big" / "frame.npy"), frame[rows.astype(int)])
    assert sum(os.path.getsize(p) for p in (tmp_path / "big").iterdir()) <= 1 << 20
