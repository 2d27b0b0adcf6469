"""Hit frames (c2rt_render_hits / c2rt_render_hits_device): for every pixel the hit record c2rt_render_pixel returns for it
(node, distance, unit normal, uv, rounded to FP32), from one launch per band, with no colour and no side effect on the colour
frames, the ray counters or the cancel flag.  The pixel pick is the reference the planes are checked against, pixel by pixel."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import chess2rt_b200 as c2
from chess2rt_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SC = os.path.join(ROOT, "scenes")
TSC = os.path.join(ROOT, "tests", "scenes")
EXE = os.path.join(ROOT, "chess2rt_b200", "chess2rt_headless")
HAS_GPU = c2.device_count() > 0
PLANES = ("node", "dist", "normal", "uv")
GI_MESSAGE = "pixel pick on a GI frame"


@pytest.fixture(scope="module")
def ctx():
    c2.init(1, [0])
    yield
    c2.shutdown()


def big_scene_text(n_side, width, height):
    """n_side x n_side pieces (spheres, cubes, a CSG of both, every third one scaled) on a checker floor: n_side^2 + 1 nodes,
    beyond the constant scene block for n_side = 16."""
    geoms = ['Plane "floor" { y 0 }', 'Sphere "s" { center 0 0 0; R 4 }', 'Cube "c" { center 0 0 0; side 7 }',
             'Sphere "cut" { center 2 2 -2; R 3.5 }', 'CsgDiff "d" { left "c"; right "cut" }', 'CsgUnion "u" { left "s"; right "c" }']
    nodes = ['Node "floor" { geometry "floor"; shader "f" }']
    for k in range(n_side * n_side):
        i, j = divmod(k, n_side)
        scale = "scale 1.3 0.8 1.1; " if k % 3 == 0 else ""
        nodes.append('Node "n%d" { geometry "%s"; shader "%s"; %stranslate %g %g %g }'
                     % (k, "scdu"[k % 4], "abp"[k % 3], scale, (i - n_side / 2) * 12.0, 4.0 + (k % 5), (j - n_side / 2) * 12.0))
    return ('Scene { GlobalSettings { frameWidth %d; frameHeight %d; ambientLightColor 0.1 0.1 0.12; AAEnabled true; prepassEnabled false }\n'
            ' Camera { pos 5 %g %g; yaw 8; pitch -32; roll 2; fov 70 }\n'
            ' Lights { PointLight "l" { pos -150 260 -120; color 1 0.95 0.9; power 70000 } }\n'
            ' Geometries { %s }\n Textures { Checker "chk" { color1 0.15 0.15 0.2; color2 0.9 0.85 0.8; size 9 } }\n'
            ' Shaders { Lambert "f" { color 1 1 1; texture "chk" }; Lambert "a" { color 0.8 0.4 0.3 }; Lambert "b" { color 0.3 0.7 0.4 }; '
            'Phong "p" { color 0.3 0.4 0.9; exponent 30; strength 0.6 } }\n'
            ' Nodes { %s } }\n') % (width, height, 9.0 * n_side, -10.0 * n_side, "; ".join(geoms), "; ".join(nodes))


def pick_planes(g, seed=0):
    """c2rt_render_pixel for every pixel, with the camera and settings blocks a hit frame of the same seed gets."""
    w, h = g.frame_size
    cam, st = g.frame_blocks(seed=seed)
    handle = g.device_scene()
    out = {"node": np.empty((h, w), np.int32), "dist": np.empty((h, w)), "normal": np.empty((h, w, 3)), "uv": np.empty((h, w, 2))}
    rgb, hit = (C.c_float * 3)(), api.Hit()
    for y in range(h):
        for x in range(w):
            assert api.lib.c2rt_render_pixel(handle, C.byref(cam), C.byref(st), x, y, rgb, C.byref(hit)) == 0
            out["node"][y, x] = hit.node
            out["dist"][y, x] = hit.dist
            out["normal"][y, x] = list(hit.normal)
            out["uv"][y, x] = (hit.u, hit.v)
    return out


def _ordered(a):
    i = np.asarray(a, np.float32).view(np.int32).astype(np.int64)
    return np.where(i < 0, -(i & 0x7fffffff), i)   # monotone in the float value; -0 and +0 map to 0


def assert_within_ulp(got, ref, what):
    """got (float32) within one FP32 ulp of the FP32 rounding of ref (float64); +inf only where ref rounds to +inf."""
    with np.errstate(over="ignore"):   # a miss's 1e99 rounds to +inf
        r32 = np.asarray(ref).astype(np.float32)
    same_inf = np.isinf(got) == np.isinf(r32)
    assert same_inf.all(), (what, np.argwhere(~same_inf)[:5])
    fin = ~np.isinf(r32)
    ulps = np.abs(_ordered(got[fin]) - _ordered(r32[fin]))
    assert ulps.max(initial=0) <= 1, (what, int(ulps.max()), int((ulps > 0).sum()))


def assert_planes_match_pick(planes, pick, what):
    assert np.array_equal(planes["node"], pick["node"]), (what, np.argwhere(planes["node"] != pick["node"])[:5])
    assert_within_ulp(planes["dist"], pick["dist"], f"{what}: dist")
    # normal and uv of hits only: after a miss the pixel pick's record keeps the normal and uv of the pick before it
    hit = pick["node"] >= 0
    for name in ("normal", "uv"):
        assert_within_ulp(planes[name][hit], pick[name][hit], f"{what}: {name}")
    miss = ~hit
    assert np.isposinf(planes["dist"][miss]).all()
    assert (planes["normal"][miss] == 0).all() and (planes["uv"][miss] == 0).all()


def scene(path, size=None, **over):
    g = c2.HostScene(path)
    if size:
        g.set_frame_size(*size)
    g.override(**over)
    return g


CASES = [
    ("lecture4", os.path.join(SC, "lecture4.sdl"), (97, 61), {}),
    ("lecture4-proc-texture", os.path.join(SC, "lecture4-proc-texture.sdl"), (97, 61), {}),
    ("lecture5", os.path.join(SC, "lecture5.sdl"), (97, 61), {}),
    ("chessboard", os.path.join(SC, "chessboard.sdl"), (96, 54), {}),
    ("quirks", os.path.join(TSC, "quirks.sdl"), (97, 61), {}),
    ("nested", os.path.join(TSC, "nested.sdl"), (97, 61), {}),
    ("sky", os.path.join(TSC, "sky.sdl"), (97, 61), {}),
    ("sky_plane", os.path.join(TSC, "sky_plane.sdl"), (97, 61), {}),
    ("stereo_dof", os.path.join(TSC, "stereo_dof.sdl"), (97, 61), {}),
    ("zaphod_dof", os.path.join(SC, "zaphod.sdl"), (97, 61), {"dof": 1, "num_samples": 3}),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,path,size,over", CASES, ids=[c[0] for c in CASES])
def test_every_pixel_equals_the_pixel_pick(ctx, name, path, size, over):
    g = scene(path, size, **over)
    seed = 11 if over.get("dof") or "stereo" in name else 0
    planes, st = g.render_hits(seed=seed)
    assert st.launches >= 1 and st.n_gpus == 1
    assert_planes_match_pick(planes, pick_planes(g, seed), name)
    assert (planes["node"] >= 0).any()


@pytest.mark.gpu
def test_every_pixel_of_a_scene_beyond_the_constant_block(ctx, tmp_path):
    p = tmp_path / "big.sdl"
    p.write_text(big_scene_text(16, 97, 61))
    g = c2.HostScene(str(p))
    assert g.info()["nodes"] == 257
    planes, _ = g.render_hits()
    assert_planes_match_pick(planes, pick_planes(g), "257 nodes")
    assert len(np.unique(planes["node"])) > 20


@pytest.mark.gpu
@pytest.mark.parametrize("solo_fast", [True, False])
def test_one_plane_camera_with_roll(ctx, monkeypatch, solo_fast):
    """A rolled camera over the one-plane scene: the regular plane test (solo_plane_test) and, with the regular path turned
    off (C2RT_NO_SOLO_FAST=1, read per frame), the general one (node_exact)."""
    if not solo_fast:
        monkeypatch.setenv("C2RT_NO_SOLO_FAST", "1")
    for path in (os.path.join(SC, "lecture4.sdl"), os.path.join(SC, "zaphod.sdl")):
        g = scene(path, (97, 61), dof=0)
        g.camera_rotate(7.0, 23.0, -4.0)
        planes, _ = g.render_hits()
        assert_planes_match_pick(planes, pick_planes(g), f"{path} rolled")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["quirks.sdl", "nested.sdl"])
def test_node_plane_equals_the_oracle(ctx, name):
    from oracle_binding import OracleScene
    path = os.path.join(TSC, name)
    g, o = scene(path, (64, 40)), OracleScene(path)
    o.set_frame_size(64, 40)
    planes, _ = g.render_hits(planes=("node",))
    assert set(planes) == {"node"}
    ref = np.array([[int(o.render_pixel(x, y)[1][0]) for x in range(64)] for y in range(40)], np.int32)
    assert np.array_equal(planes["node"], ref), np.argwhere(planes["node"] != ref)[:5]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["lecture5.sdl", "../tests/scenes/nested.sdl", "../tests/scenes/stereo_dof.sdl"])
def test_global_memory_form_gives_the_same_planes(ctx, monkeypatch, name):
    const, _ = scene(os.path.join(SC, name), (97, 61)).render_hits(seed=5)
    monkeypatch.setenv("C2RT_FORCE_GLOBAL", "1")   # read at scene-create time
    glob, _ = scene(os.path.join(SC, name), (97, 61)).render_hits(seed=5)
    for k in PLANES:
        assert np.array_equal(const[k], glob[k]), k


def _device_planes(torch, h, w):
    return {"node": torch.full((h, w), 7, dtype=torch.int32, device="cuda"),
            "dist": torch.full((h, w), 7.0, device="cuda"),
            "normal": torch.full((h, w, 3), 7.0, device="cuda"),
            "uv": torch.full((h, w, 2), 7.0, device="cuda")}


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["lecture5.sdl", "lecture4.sdl", "../tests/scenes/stereo_dof.sdl"])
@pytest.mark.parametrize("n_ranks", [2, 3])
@pytest.mark.parametrize("compact", [0, 1])
def test_emulated_bands_reassemble_to_the_one_rank_planes(ctx, name, n_ranks, compact):
    import torch
    g = scene(os.path.join(SC, name), (97, 61))
    ref, _ = g.render_hits(seed=2)
    w, h = g.frame_size
    cam, st = g.frame_blocks(seed=2)
    handle = g.device_scene()
    band_rows = 16
    got = {k: np.zeros_like(v) for k, v in ref.items()}
    for r in range(n_ranks):
        rows = [y for y in range(h) if (y // band_rows) % n_ranks == r]
        assert len(rows) == c2.band_rows_owned(h, r, n_ranks, band_rows)
        out = _device_planes(torch, len(rows) if compact else h, w)
        band = api.Band(r, n_ranks, band_rows, compact)
        api.render_hits_device(handle, cam, st, *(out[k].data_ptr() for k in PLANES), band=band)
        torch.cuda.synchronize()
        for k in PLANES:
            a = out[k].cpu().numpy()
            got[k][rows] = a[:len(rows)] if compact else a[rows]
    for k in PLANES:
        assert np.array_equal(got[k].view(np.uint32), ref[k].view(np.uint32)), k


@pytest.mark.gpu
def test_two_devices_give_the_one_device_planes():
    if c2.device_count() < 2:
        pytest.skip("needs two GPUs")
    path = os.path.join(SC, "lecture5.sdl")
    c2.init(1, [0])
    try:
        one, _ = scene(path, (197, 161)).render_hits()
        c2.init(2)
        two, st = scene(path, (197, 161)).render_hits()
        assert st.n_gpus == 2
        for k in PLANES:
            assert np.array_equal(one[k].view(np.uint32), two[k].view(np.uint32)), k
    finally:
        c2.shutdown()


@pytest.mark.gpu
def test_device_planes_on_a_side_stream(ctx):
    import torch
    g = scene(os.path.join(SC, "chessboard.sdl"), (96, 54))
    ref, _ = g.render_hits()
    w, h = g.frame_size
    cam, st = g.frame_blocks()
    handle = g.device_scene()
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        out = _device_planes(torch, h, w)
    api.render_hits_device(handle, cam, st, *(out[k].data_ptr() for k in PLANES), stream=stream.cuda_stream)
    stream.synchronize()
    for k in PLANES:
        assert np.array_equal(out[k].cpu().numpy().view(np.uint32), ref[k].view(np.uint32)), k
    # only the node plane: it is written with guard words on both sides, the other planes are not touched
    guard = 64
    with torch.cuda.stream(stream):
        buf = torch.full((h * w + 2 * guard,), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
        others = _device_planes(torch, h, w)
    api.render_hits_device(handle, cam, st, node=buf.data_ptr() + 4 * guard, stream=stream.cuda_stream)
    stream.synchronize()
    b = buf.cpu().numpy()
    assert (b[:guard] == 0x5A5A5A5A).all() and (b[-guard:] == 0x5A5A5A5A).all()
    assert np.array_equal(b[guard:-guard].reshape(h, w), ref["node"])
    for k in ("dist", "normal", "uv"):
        assert (others[k].cpu().numpy() == 7).all(), k


@pytest.mark.gpu
def test_hit_frames_leave_colour_frames_counters_and_cancel_alone(ctx):
    g = scene(os.path.join(SC, "lecture5.sdl"), (97, 61))
    before, argb0, st0 = g.render(argb=True, count_rays=True)
    handle = g.device_scene()
    assert api.read_ray_counters(handle) == (0, 0)   # (c2rt_render has read and zeroed them)
    cam, st = g.frame_blocks(count_rays=True)
    assert st.count_rays == 1
    planes, hst = g.render_hits()
    import torch
    node = torch.empty((61, 97), dtype=torch.int32, device="cuda")
    api.render_hits_device(handle, cam, st, node=node.data_ptr())
    torch.cuda.synchronize()
    assert api.read_ray_counters(handle) == (0, 0)
    api.cancel()   # no frame in progress: cancels nothing, and a hit frame neither takes nor leaves the request
    planes2, _ = g.render_hits()
    after, argb1, st1 = g.render(argb=True, count_rays=True)
    assert not g.cancelled
    assert np.array_equal(before.view(np.uint32), after.view(np.uint32)) and np.array_equal(argb0, argb1)
    assert (st0.primary_rays, st0.shadow_rays) == (st1.primary_rays, st1.shadow_rays)
    for k in PLANES:
        assert np.array_equal(planes[k].view(np.uint32), planes2[k].view(np.uint32)), k


@pytest.mark.gpu
def test_errors(ctx):
    g = scene(os.path.join(SC, "lecture4.sdl"), (64, 48))   # (no Phong shader: GI frames of it pass the frame checks)
    handle = g.device_scene()
    cam, st = g.frame_blocks()
    node = np.empty((48, 64), np.int32)
    p = api.HitPlanes(node.ctypes.data, None, None, None)
    gi = api.Settings.from_buffer_copy(st)
    gi.gi_enabled, gi.paths_per_pixel = 1, 4
    assert api.lib.c2rt_render_hits(handle, C.byref(cam), C.byref(gi), C.byref(p), None) == -2
    assert GI_MESSAGE in api.lib.c2rt_last_error().decode()
    assert api.lib.c2rt_render_pixel(handle, C.byref(cam), C.byref(gi), 0, 0, (C.c_float * 3)(), None) == -2
    assert api.lib.c2rt_render_hits_device(handle, C.byref(cam), C.byref(gi), None, C.byref(p), None, None) == -2
    assert GI_MESSAGE in api.lib.c2rt_last_error().decode()
    empty = api.HitPlanes()
    assert api.lib.c2rt_render_hits(handle, C.byref(cam), C.byref(st), C.byref(empty), None) == -1
    assert api.lib.c2rt_render_hits_device(handle, C.byref(cam), C.byref(st), None, C.byref(empty), None, None) == -1
    assert api.lib.c2rt_render_hits(handle, C.byref(cam), C.byref(st), None, None) == -1
    flags = C.c_uint32 * 4
    band = api.Band(0, 2, 8, 0, C.cast(C.pointer(flags()), C.c_void_p), 1)
    assert api.lib.c2rt_render_hits_device(handle, C.byref(cam), C.byref(st), C.byref(band), C.byref(p), None, None) == -1
    assert "done_flags" in api.lib.c2rt_last_error().decode()
    with pytest.raises(ValueError):
        g.render_hits(planes=("depth",))


@pytest.mark.gpu
def test_both_device_entry_points_refuse_a_malformed_band_alike(ctx):
    import torch
    g = scene(os.path.join(SC, "lecture4.sdl"), (64, 48))
    handle = g.device_scene()
    cam, st = g.frame_blocks()
    rgb = torch.zeros((48, 64, 3), device="cuda")
    node = torch.zeros((48, 64), dtype=torch.int32, device="cuda")
    p = api.HitPlanes(node.data_ptr(), None, None, None)
    # no ranks, a rank beyond them, empty bands, bands of a partial tile
    for rank, n_ranks, band_rows in [(0, 0, 8), (2, 2, 8), (0, 1, 0), (1, 2, 12)]:
        band = api.Band(rank, n_ranks, band_rows, 0)
        assert api.lib.c2rt_render_device(handle, C.byref(cam), C.byref(st), C.byref(band), rgb.data_ptr(), None, None, None) == -1
        colour = api.lib.c2rt_last_error().decode()
        assert colour == f"bad band (rank {rank} of {n_ranks}, band_rows {band_rows}; band_rows must be a multiple of 8)"
        assert api.lib.c2rt_render_hits_device(handle, C.byref(cam), C.byref(st), C.byref(band), C.byref(p), None, None) == -1
        assert api.lib.c2rt_last_error().decode() == colour
    torch.cuda.synchronize()
    assert (rgb.cpu().numpy() == 0).all() and (node.cpu().numpy() == 0).all()


def _read_pfm1(path):
    magic, dims, scale, body = open(path, "rb").read().split(b"\n", 3)
    w, h = map(int, dims.split())
    assert magic == b"Pf" and float(scale) < 0   # little endian
    return np.frombuffer(body, "<f4").reshape(h, w)[::-1]


def _read_pgm16(path):
    data = open(path, "rb").read()
    magic, dims, maxval, body = data.split(b"\n", 3)
    w, h = map(int, dims.split())
    assert magic == b"P5" and maxval == b"65535"
    return np.frombuffer(body, ">u2").reshape(h, w)


@pytest.mark.gpu
def test_command_line_depth_and_ids(tmp_path):
    d, i = tmp_path / "d.pfm", tmp_path / "ids.pgm"
    path = os.path.join(SC, "lecture5.sdl")
    r = subprocess.run([EXE, "--file", path, "--width", "64", "--height", "48", "--depth", str(d), "--ids", str(i)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    c2.init(1, [0])
    try:
        planes, _ = scene(path, (64, 48)).render_hits(planes=("node", "dist"))
    finally:
        c2.shutdown()
    assert np.array_equal(_read_pfm1(d).view(np.uint32), planes["dist"].view(np.uint32))
    assert np.array_equal(_read_pgm16(i).astype(np.int32) - 1, planes["node"])


@pytest.mark.skipif(HAS_GPU, reason="checks the failure without a GPU")
def test_without_a_gpu_both_paths_fail_with_a_cuda_error(tmp_path):
    g = c2.HostScene(os.path.join(SC, "lecture4.sdl"))
    with pytest.raises(c2.C2rtError) as e:
        g.render_hits()
    assert e.value.status == -3
    with pytest.raises(c2.C2rtError) as e:   # a device scene for c2rt_render_hits_device cannot be made either
        g.device_scene()
    assert e.value.status == -3
    d, i = tmp_path / "d.pfm", tmp_path / "ids.pgm"
    r = subprocess.run([EXE, "--file", os.path.join(SC, "lecture4.sdl"), "--width", "64", "--height", "48", "--depth", str(d),
                        "--ids", str(i)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 1 and "CUDA" in r.stderr and not d.exists() and not i.exists()


def test_hit_plane_bindings_follow_the_header():
    header = open(os.path.join(ROOT, "include", "c2rt.h")).read()
    assert "typedef struct c2rt_hit_planes" in header
    assert C.sizeof(api.HitPlanes) == 4 * 8
    assert list(api.HIT_PLANES) == [f[0] for f in api.HitPlanes._fields_] == list(PLANES)
    assert {"c2rt_render_hits", "c2rt_render_hits_device"} <= set(api.C_ABI_SYMBOLS)
    r = subprocess.run([EXE], capture_output=True, text=True, timeout=60)
    assert r.returncode == 2 and "--depth" in r.stderr and "--ids" in r.stderr
