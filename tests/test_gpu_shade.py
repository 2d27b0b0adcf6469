"""Shaded ray queries (c2rt_shade_rays / c2rt_shade_rays_device): the colour Renderer.trace returns for caller-supplied rays,
one launch per device, checked against the CPU oracle's trace (tests/oracle_shade.cpp with tests/oracle_rays.cpp, built here
against oracle/), against the product's own AA-off colour frames, and against themselves through every route and query order."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import chess2rt_b200 as c2
from chess2rt_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SC = os.path.join(ROOT, "scenes")
TSC = os.path.join(ROOT, "tests", "scenes")
HAS_GPU = c2.device_count() > 0
N_PER_GEN = 17000   # three generators: about 50k queries per scene
TIE = 1e-9          # the oracle's near-tie threshold (relative gap)


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


# ---------------------------------------------------------------- the oracle's trace
@pytest.fixture(scope="module")
def oracle_shade(tmp_path_factory):
    """path -> (o, d) -> (rgb [n, 3] float64, gap [n]): orc::Renderer::trace, and the near-tie gap of its camera hit and
    shadow segments."""
    cxx = os.environ.get("CXX") or shutil.which("g++") or "g++"
    so = str(tmp_path_factory.mktemp("orr") / "liborr.so")
    subprocess.run([cxx, "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-pthread", "-shared", "-I", os.path.join(ROOT, "oracle"),
                    "-o", so, os.path.join(ROOT, "tests", "oracle_rays.cpp"), os.path.join(ROOT, "tests", "oracle_shade.cpp")],
                   check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.orr_last_error.restype = C.c_char_p
    lib.orr_scene_load.restype = C.c_void_p
    lib.orr_scene_load.argtypes = [C.c_char_p]
    lib.orr_scene_free.argtypes = [C.c_void_p]
    lib.orr_scene_free.restype = None
    lib.orr_shade_rays.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.orr_shade_rays.restype = None

    def shade(path, o, d):
        h = lib.orr_scene_load(os.fspath(path).encode())
        if not h:
            raise RuntimeError(lib.orr_last_error().decode())
        try:
            o, d = np.ascontiguousarray(o, np.float64), np.ascontiguousarray(d, np.float64)
            out = np.empty((len(o), 4))
            lib.orr_shade_rays(h, len(o), o.ctypes.data, d.ctypes.data, out.ctypes.data)
        finally:
            lib.orr_scene_free(h)
        return out[:, :3], out[:, 3]
    return shade


@pytest.fixture(scope="module")
def ctx():
    c2.init(1, [0])
    yield
    c2.shutdown()


@pytest.fixture(scope="module")
def big_path(tmp_path_factory):
    p = tmp_path_factory.mktemp("big") / "big.sdl"
    p.write_text(big_scene_text(16, 160, 100))
    return str(p)


# ---------------------------------------------------------------- query generators (seeded)
def camera_vectors(g):
    """pos, upLeft - pos, upRight - upLeft, downLeft - upLeft of the scene camera after beginFrame (c2rt_camera)."""
    cam, _ = g.frame_blocks()
    pos, ul, ur, dl = (np.array(v[:]) for v in (cam.pos, cam.up_left, cam.up_right, cam.down_left))
    return pos, ul - pos, ur - ul, dl - ul


def camera_rays(g, w, h):
    """The ray through the top-left corner of every pixel of a w x h frame, in row order (the AA-off camera ray of a frame)."""
    pos, ul, du, dv = camera_vectors(g)
    ys, xs = np.mgrid[0:h, 0:w]
    sx, sy = xs.reshape(-1, 1) * (1.0 / w), ys.reshape(-1, 1) * (1.0 / h)
    d = dv * sy + (du * sx + ul)
    return np.broadcast_to(pos, d.shape).copy(), d


def node_centres(g):
    """World-space centre of every node's primitive (translation + the primitive's centre; a CSG's translation)."""
    dsc = g.desc().contents
    out = []
    for i in range(dsc.n_nodes):
        off = np.array(dsc.node_offset[3 * i:3 * i + 3])
        gi = dsc.node_geom[i]
        c = np.array(dsc.geom_params[4 * gi:4 * gi + 3]) if dsc.geom_type[gi] in (1, 2) else np.zeros(3)
        out.append(off + c)
    return np.array(out)


def scene_box(g):
    pts = np.vstack([node_centres(g), camera_vectors(g)[0][None]])
    lo, hi = pts.min(0), pts.max(0)
    pad = 0.2 * (hi - lo) + 1.0
    return lo - pad, hi + pad


def all_queries(g, seed=0):
    """Camera rays in row order, random rays in a box around the scene, rays aimed near node centres.  The frame is an odd
    number of pixels wide and the aim points are jittered by 1 % of the box: a symmetric camera's centre column, or a ray
    aimed exactly at a plane's offset or a CSG's centre, lands on a checker or bitmap cell edge or a crossing tie, where the
    reference's own colour is discontinuous."""
    w = 157
    o1, d1 = camera_rays(g, w, N_PER_GEN // w)
    rng = np.random.default_rng(seed)
    lo, hi = scene_box(g)
    o2, d2 = rng.uniform(lo, hi, (N_PER_GEN, 3)), rng.normal(size=(N_PER_GEN, 3))
    cen = node_centres(g)
    o3 = rng.uniform(lo, hi, (N_PER_GEN, 3))
    aim = cen[rng.integers(0, len(cen), N_PER_GEN)] + rng.normal(scale=0.01 * np.linalg.norm(hi - lo), size=(N_PER_GEN, 3))
    d3 = aim - o3
    return np.vstack([o1, o2, o3]), np.vstack([d1, d2, d3])


def pack_argb(rgb):
    """Color.toRGB32 (color.d:154-162) through c2rt_srgb_table with the kernel's lut8 rule (color.d:209-214)."""
    lut = api.srgb_table().astype(np.uint32)
    x = np.ascontiguousarray(rgb, np.float32)
    idx = np.clip((x * np.float32(4096.0)).astype(np.int64), 0, 4096)
    v = np.where(x <= 0, 0, np.where(x >= 1, 255, lut[idx])).astype(np.uint32)
    return v[..., 2] | (v[..., 1] << 8) | (v[..., 0] << 16)


def channels(argb):
    return np.stack([(argb >> 16) & 0xFF, (argb >> 8) & 0xFF, argb & 0xFF], axis=1).astype(np.int32)


def ambient_of(g):
    return list(g.frame_blocks()[1].ambient_light)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint8)


SCENES = [("lecture4", os.path.join(SC, "lecture4.sdl")), ("lecture4-proc-texture", os.path.join(SC, "lecture4-proc-texture.sdl")),
          ("lecture5", os.path.join(SC, "lecture5.sdl")), ("chessboard", os.path.join(SC, "chessboard.sdl")),
          ("zaphod", os.path.join(SC, "zaphod.sdl")), ("quirks", os.path.join(TSC, "quirks.sdl")),
          ("nested", os.path.join(TSC, "nested.sdl")), ("sky", os.path.join(TSC, "sky.sdl")), ("big257", None)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,path", SCENES, ids=[s[0] for s in SCENES])
def test_colours_equal_the_oracles_trace(ctx, oracle_shade, big_path, name, path):
    """About 50k queries per scene.  Every query the oracle does not flag as a near-tie is within 1e-3 of its colour; at most
    1 % are flagged, and at most 0.1 % of the queries have an 8-bit channel more than 1 LSB off.  ARGB is the packing of the returned
    rgb, bit for bit."""
    path = path or big_path
    g = c2.HostScene(path)
    if name == "big257":
        assert g.info()["nodes"] == 257
    o, d = all_queries(g)
    rgb, argb, st = g.shade_rays(o, d, argb=True)
    assert st.launches == 1 and st.n_gpus == 1
    assert rgb.shape == (len(o), 3) and rgb.dtype == np.float32 and argb.dtype == np.uint32
    assert np.array_equal(argb, pack_argb(rgb)), name
    ref, gap = oracle_shade(path, o, d)
    flagged = gap < TIE
    # (flagged: 0 on six scenes; 0.3-0.5 % on chessboard, quirks and sky, whose coincident surfaces — piece bases flush with the
    # board — the rays aimed near node centres meet with gaps of exactly 0 or a few ulps)
    assert flagged.mean() <= 1e-2, (name, int(flagged.sum()))
    err = np.abs(rgb.astype(np.float64) - ref).max(axis=1)
    worst = float(err[~flagged].max(initial=0))
    print(f"{name}: largest |rgb - oracle| {worst:.3g} over {int((~flagged).sum())} queries, {int(flagged.sum())} flagged")
    assert worst <= 1e-3, (name, worst, np.argwhere(err > 1e-3)[:5].ravel())
    lsb = np.abs(channels(argb) - channels(pack_argb(ref)))
    assert (lsb > 1).any(axis=1).mean() <= 1e-3, (name, int((lsb > 1).any(axis=1).sum()))
    assert (rgb.max(axis=1) > 0).mean() > 0.2, name
    if name == "sky":   # misses take the cubemap's colour (the environment extension): many queries see the sky
        miss = g.trace_rays(o, d, planes=("node",))[0]["node"] < 0
        assert (rgb[miss].max(axis=1) > 0).sum() > 1000


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(96, 64), (97, 61)], ids=["96x64", "97x61"])
@pytest.mark.parametrize("which", ["lecture4", "lecture5", "chessboard", "big257"])
def test_pixel_corner_rays_reproduce_the_aa_off_colour_frame(ctx, oracle_shade, big_path, which, size):
    path = big_path if which == "big257" else os.path.join(SC, which + ".sdl")
    w, h = size
    g = c2.HostScene(path)
    g.set_frame_size(w, h)
    g.override(aa=0, dof=0)
    frame, fargb, _ = g.render(argb=True)
    o, d = camera_rays(g, w, h)
    rgb, argb, _ = g.shade_rays(o, d, argb=True)
    diff = np.abs(rgb - frame.reshape(-1, 3)).max(axis=1)
    off = diff > 1e-5
    print(f"{which} {w}x{h}: largest |ray - frame| {diff.max():.3g}, {int(off.sum())} pixels over 1e-5")
    assert off.mean() <= 1e-4, (which, int(off.sum()))
    if off.any():   # a silhouette or shadow-edge pixel: its ray and the frame's camera ray part on the node or at a tie
        node = g.trace_rays(o[off], d[off], planes=("node",))[0]["node"]
        hits, _ = g.render_hits(planes=("node",))
        _, gap = oracle_shade(path, o[off], d[off])
        assert ((node != hits["node"].reshape(-1)[off]) | (gap < TIE)).all(), (which, np.argwhere(off).ravel()[:5])
    assert (argb == fargb.reshape(-1)).mean() >= 0.999, which


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["chessboard", "big257"])
def test_colours_do_not_depend_on_order_or_batch(ctx, big_path, which):
    path = big_path if which == "big257" else os.path.join(SC, "chessboard.sdl")
    g = c2.HostScene(path)
    (o1, d1), (o2, d2) = all_queries(g, seed=3), all_queries(g, seed=13)
    o, d = np.vstack([o1, o2]), np.vstack([d1, d2])   # > 1 + 31 + 257 + 100003 queries
    ref, aref, _ = g.shade_rays(o, d, argb=True)
    perm = np.random.default_rng(5).permutation(len(o))
    got, agot, _ = g.shade_rays(o[perm], d[perm], argb=True)
    assert np.array_equal(bits(got), bits(ref[perm])) and np.array_equal(agot, aref[perm])
    start = 0
    for n in (1, 31, 257, 100003):
        part, apart, _ = g.shade_rays(o[start:start + n], d[start:start + n], argb=True)
        assert np.array_equal(bits(part), bits(ref[start:start + n])) and np.array_equal(apart, aref[start:start + n]), n
        start += n


@pytest.mark.gpu
def test_global_memory_form_gives_the_same_bits(ctx, monkeypatch):
    path = os.path.join(SC, "lecture5.sdl")
    g = c2.HostScene(path)
    o, d = all_queries(g, seed=9)
    const, aconst, _ = g.shade_rays(o, d, argb=True)
    monkeypatch.setenv("C2RT_FORCE_GLOBAL", "1")   # read at scene-create time
    glob, aglob, _ = c2.HostScene(path).shade_rays(o, d, argb=True)
    assert np.array_equal(bits(const), bits(glob)) and np.array_equal(aconst, aglob)


@pytest.mark.gpu
def test_rgb_only_argb_only_and_both_give_the_same_bits(ctx):
    g = c2.HostScene(os.path.join(SC, "lecture5.sdl"))
    o, d = all_queries(g, seed=8)
    o, d = o[:-3], d[:-3]
    ref, aref, _ = g.shade_rays(o, d, argb=True)
    handle, amb = g.device_scene(), (C.c_float * 3)(*ambient_of(g))
    n = len(o)
    rgb = np.full((n, 3), 7.0, np.float32)
    argb = np.full(n, 7, np.uint32)
    st = api.Stats()
    assert api.lib.c2rt_shade_rays(handle, amb, n, o.ctypes.data, d.ctypes.data, rgb.ctypes.data, None, C.byref(st)) == 0
    assert np.array_equal(bits(rgb), bits(ref)) and st.launches == 1
    assert api.lib.c2rt_shade_rays(handle, amb, n, o.ctypes.data, d.ctypes.data, None, argb.ctypes.data, C.byref(st)) == 0
    assert np.array_equal(argb, aref)


@pytest.mark.gpu
def test_device_entry_point_on_a_side_stream_with_guard_words(ctx):
    import torch
    g = c2.HostScene(os.path.join(SC, "chessboard.sdl"))
    o, d = all_queries(g, seed=4)
    n = len(o) - 5   # a ragged tail
    o, d = o[:n], d[:n]
    ref, aref, _ = g.shade_rays(o, d, argb=True)
    handle = g.device_scene()
    stream = torch.cuda.Stream()
    guard = 64
    with torch.cuda.stream(stream):
        to, td = (torch.from_numpy(a).to("cuda") for a in (o, d))
        rgb = torch.full((3 * n + 2 * guard,), 7.0, dtype=torch.float32, device="cuda")
        argb = torch.full((n + 2 * guard,), 7, dtype=torch.int32, device="cuda")
    api.shade_rays_device(handle, n, to.data_ptr(), td.data_ptr(), ambient_of(g), d_rgb=rgb.data_ptr() + 4 * guard,
                          d_argb=argb.data_ptr() + 4 * guard, stream=stream.cuda_stream)
    stream.synchronize()
    r, a = rgb.cpu().numpy(), argb.cpu().numpy().view(np.uint32)
    assert (r[:guard] == 7).all() and (r[-guard:] == 7).all() and (a[:guard] == 7).all() and (a[-guard:] == 7).all()
    assert np.array_equal(bits(r[guard:-guard]), bits(ref.reshape(-1))) and np.array_equal(a[guard:-guard], aref)
    # an rgb plane 4 bytes off 16-byte alignment: full CTAs store per query there
    api.shade_rays_device(handle, n, to.data_ptr(), td.data_ptr(), ambient_of(g), d_rgb=rgb.data_ptr() + 4 * (guard + 1),
                          stream=stream.cuda_stream)
    stream.synchronize()
    r = rgb.cpu().numpy()
    assert np.array_equal(bits(r[guard + 1:guard + 1 + 3 * n]), bits(ref.reshape(-1)))


@pytest.mark.gpu
def test_two_devices_give_the_one_device_bits():
    if c2.device_count() < 2:
        pytest.skip("needs two GPUs")
    path = os.path.join(SC, "chessboard.sdl")
    c2.init(1, [0])
    try:
        g = c2.HostScene(path)
        o, d = all_queries(g)
        one, a1, _ = g.shade_rays(o, d, argb=True)
        c2.init(2)
        g = c2.HostScene(path)
        two, a2, st = g.shade_rays(o, d, argb=True)
        assert st.n_gpus == 2 and st.launches == 2
        assert np.array_equal(bits(one), bits(two)) and np.array_equal(a1, a2)
    finally:
        c2.shutdown()


@pytest.mark.gpu
def test_untraced_queries_are_black_even_under_a_cubemap(ctx):
    g = c2.HostScene(os.path.join(TSC, "sky.sdl"))
    nan, inf = float("nan"), float("inf")
    o = np.array([[0, 5, 0], [nan, 5, 0], [0, 5, 0], [inf, 5, 0], [0, 5, 0], [0, 5, 0], [0, 5, 0], [0, -inf, 0]], np.float64)
    d = np.array([[0, 0, 0], [0, 1, 0], [0, nan, 0], [0, 1, 0], [-inf, 1, 0], [1e-200, 0, 0], [0, 1e300, 0], [0, 1, 0]], np.float64)
    rgb, argb, _ = g.shade_rays(o, d, argb=True)
    assert (rgb == 0).all() and (argb == 0).all()
    sky, skyargb, _ = g.shade_rays(np.array([[0.0, 5.0, 0.0]]), np.array([[0.1, 1.0, 0.2]]), argb=True)
    assert (sky > 0).any() and skyargb[0] != 0   # the same origin, traced: the cubemap's colour


@pytest.mark.gpu
def test_queries_leave_colour_frames_counters_and_cancel_alone(ctx):
    g = c2.HostScene(os.path.join(SC, "lecture5.sdl"))
    g.set_frame_size(97, 61)
    before, argb0, st0 = g.render(argb=True, count_rays=True)
    handle = g.device_scene()
    assert api.read_ray_counters(handle) == (0, 0)
    o, d = all_queries(g)
    r1, a1, _ = g.shade_rays(o, d, argb=True)
    assert api.read_ray_counters(handle) == (0, 0)
    api.cancel()   # no frame in progress: cancels nothing, and a query neither takes nor leaves the request
    r2, a2, _ = g.shade_rays(o, d, argb=True)
    after, argb1, st1 = g.render(argb=True, count_rays=True)
    assert not g.cancelled
    assert np.array_equal(before.view(np.uint32), after.view(np.uint32)) and np.array_equal(argb0, argb1)
    assert (st0.primary_rays, st0.shadow_rays) == (st1.primary_rays, st1.shadow_rays)
    assert np.array_equal(bits(r1), bits(r2)) and np.array_equal(a1, a2)


@pytest.mark.gpu
def test_queries_interleaved_with_colour_frames_of_another_scene(ctx):
    a = c2.HostScene(os.path.join(SC, "chessboard.sdl"))
    b = c2.HostScene(os.path.join(SC, "lecture5.sdl"))
    b.set_frame_size(64, 48)
    o, d = all_queries(a, seed=12)
    ref, aref, _ = a.shade_rays(o, d, argb=True)
    frame0, _, _ = b.render()
    for _ in range(2):
        got, agot, _ = a.shade_rays(o, d, argb=True)
        frame, _, _ = b.render()
        assert np.array_equal(bits(got), bits(ref)) and np.array_equal(agot, aref)
        assert np.array_equal(frame.view(np.uint32), frame0.view(np.uint32))


# ---------------------------------------------------------------- no GPU needed
BOGUS = C.c_void_p(16)   # never dereferenced: the argument checks come first


def test_argument_errors_come_before_any_device():
    o = np.zeros((4, 3))
    rgb = np.zeros((4, 3), np.float32)
    argb = np.zeros(4, np.uint32)
    amb = (C.c_float * 3)(0.1, 0.1, 0.1)
    L = api.lib
    for f, tail in ((L.c2rt_shade_rays, (None,)), (L.c2rt_shade_rays_device, (None, None))):
        assert f(None, None, 4, o.ctypes.data, o.ctypes.data, rgb.ctypes.data, None, *tail) == -1
        assert "scene is null" in L.c2rt_last_error().decode()
        assert f(BOGUS, None, 4, None, None, None, None, *tail) == -1
        assert "ambient is null" in L.c2rt_last_error().decode()
        assert f(BOGUS, amb, 2 ** 31, None, None, None, None, *tail) == -1
        assert "output is null" in L.c2rt_last_error().decode()
        assert f(BOGUS, amb, 2 ** 31, None, None, rgb.ctypes.data, None, *tail) == -5
        assert f(BOGUS, amb, 4, None, o.ctypes.data, None, argb.ctypes.data, *tail) == -1
        assert "input array is null" in L.c2rt_last_error().decode()
        assert f(BOGUS, amb, 4, o.ctypes.data, None, rgb.ctypes.data, argb.ctypes.data, *tail) == -1
        # n == 0: a no-op (the inputs may then be null) that zeroes stats
        st = api.Stats(kernel_ms=5.0, total_ms=1.0, n_gpus=3, launches=9)
        stats = (None,) * (len(tail) - 1) + (C.byref(st),)
        assert f(BOGUS, amb, 0, None, None, None, argb.ctypes.data, *stats) == 0
        assert (st.kernel_ms, st.total_ms, st.n_gpus, st.launches) == (0.0, 0.0, 0, 0)


@pytest.mark.skipif(HAS_GPU, reason="checks the failure without a GPU")
def test_without_a_gpu_valid_queries_fail_with_a_cuda_error():
    o = np.zeros((4, 3))
    d = np.ones((4, 3))
    rgb = np.zeros((4, 3), np.float32)
    amb = (C.c_float * 3)(0.1, 0.1, 0.1)
    assert api.lib.c2rt_shade_rays(BOGUS, amb, 4, o.ctypes.data, d.ctypes.data, rgb.ctypes.data, None, None) == -3
    g = c2.HostScene(os.path.join(SC, "lecture4.sdl"))
    with pytest.raises(c2.C2rtError) as e:
        g.shade_rays(o, d)
    assert e.value.status == -3


def test_shade_bindings_follow_the_header():
    header = open(os.path.join(ROOT, "include", "c2rt.h")).read()
    names = {"c2rt_shade_rays", "c2rt_shade_rays_device"}
    assert names <= set(api.C_ABI_SYMBOLS)
    for n in names:
        assert f"int {n}(" in header, n
        assert len(getattr(api.lib, n).argtypes) == header.split(f"int {n}(")[1].split(");")[0].count(",") + 1, n
    assert c2.shade_rays_device is api.shade_rays_device
    g = c2.HostScene(os.path.join(SC, "lecture4.sdl"))
    with pytest.raises(ValueError):
        g.shade_rays(np.zeros((3, 3)), np.zeros((2, 3)))
    with pytest.raises(ValueError):
        g.shade_rays(np.zeros((3, 2)), np.zeros((3, 2)))
