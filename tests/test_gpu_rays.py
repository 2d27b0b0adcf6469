"""Ray queries (c2rt_trace_rays / c2rt_test_visibility and their device forms): the closest hit and testVisibility of
caller-supplied rays, one launch per device, checked against the CPU oracle's two scene queries (tests/oracle_rays.cpp, built
here against oracle/), against the product's own pixel pick, and against themselves through every route and query order."""
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
RAY_PLANES = ("node", "dist", "p", "normal", "uv")
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


# ---------------------------------------------------------------- the oracle's ray queries
class OracleRays:
    def __init__(self, lib, path):
        self.lib = lib
        self._h = lib.orr_scene_load(os.fspath(path).encode())
        if not self._h:
            raise RuntimeError(lib.orr_last_error().decode())

    def __del__(self):
        if getattr(self, "_h", None):
            self.lib.orr_scene_free(self._h)

    def trace(self, o, d):
        o, d = np.ascontiguousarray(o, np.float64), np.ascontiguousarray(d, np.float64)
        out = np.empty((len(o), 11))
        self.lib.orr_trace_rays(self._h, len(o), o.ctypes.data, d.ctypes.data, out.ctypes.data)
        n = np.linalg.norm(out[:, 5:8], axis=1, keepdims=True)
        nrm = np.where(n > 0, out[:, 5:8] / np.where(n > 0, n, 1), 0)
        return {"node": out[:, 0].astype(np.int32), "dist": out[:, 1], "p": out[:, 2:5], "normal": nrm, "uv": out[:, 8:10],
                "gap": out[:, 10]}

    def visibility(self, f, t):
        f, t = np.ascontiguousarray(f, np.float64), np.ascontiguousarray(t, np.float64)
        out = np.empty((len(f), 2))
        self.lib.orr_test_visibility(self._h, len(f), f.ctypes.data, t.ctypes.data, out.ctypes.data)
        return out[:, 0].astype(bool), out[:, 1]


@pytest.fixture(scope="module")
def orr(tmp_path_factory):
    cxx = os.environ.get("CXX") or shutil.which("g++") or "g++"
    so = str(tmp_path_factory.mktemp("orr") / "liborr.so")
    subprocess.run([cxx, "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-pthread", "-shared", "-I", os.path.join(ROOT, "oracle"),
                    "-o", so, os.path.join(ROOT, "tests", "oracle_rays.cpp")], check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.orr_last_error.restype = C.c_char_p
    lib.orr_scene_load.restype = C.c_void_p
    lib.orr_scene_load.argtypes = [C.c_char_p]
    lib.orr_scene_free.argtypes = [C.c_void_p]
    lib.orr_scene_free.restype = None
    for f in (lib.orr_trace_rays, lib.orr_test_visibility):
        f.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
        f.restype = None
    return lambda path: OracleRays(lib, path)


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
    """pos, upLeft, upRight, downLeft of the scene camera after beginFrame (c2rt_camera)."""
    cam, _ = g.frame_blocks()
    return (np.array(cam.pos[:]), np.array(cam.up_left[:]), np.array(cam.up_right[:]), np.array(cam.down_left[:]))


def camera_rays(g, w, h, order="rows"):
    """The scene camera's ray directions through the pixel corners of a w x h frame: in row order, in 8x4-pixel warp order,
    or shuffled."""
    pos, ul, ur, dl = camera_vectors(g)
    ys, xs = np.mgrid[0:h, 0:w]
    if order == "patches":   # 32 consecutive queries = one 8x4 patch
        ys = ys.reshape(h // 4, 4, w // 8, 8).transpose(0, 2, 1, 3)
        xs = xs.reshape(h // 4, 4, w // 8, 8).transpose(0, 2, 1, 3)
    x, y = xs.reshape(-1, 1).astype(np.float64), ys.reshape(-1, 1).astype(np.float64)
    d = ul + (ur - ul) * (x / w) + (dl - ul) * (y / h) - pos
    o = np.broadcast_to(pos, d.shape).copy()
    if order == "shuffled":
        perm = np.random.default_rng(1).permutation(len(d))
        o, d = o[perm], d[perm]
    return o, d


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


def random_rays(g, n, seed):
    rng = np.random.default_rng(seed)
    lo, hi = scene_box(g)
    return rng.uniform(lo, hi, (n, 3)), rng.normal(size=(n, 3))


def aimed_rays(g, n, seed):
    rng = np.random.default_rng(seed)
    lo, hi = scene_box(g)
    cen = node_centres(g)
    o = rng.uniform(lo, hi, (n, 3))
    return o, cen[rng.integers(0, len(cen), n)] - o


def all_queries(g, seed=0):
    w = 160
    o1, d1 = camera_rays(g, w, N_PER_GEN // w)
    o2, d2 = random_rays(g, N_PER_GEN, seed + 1)
    o3, d3 = aimed_rays(g, N_PER_GEN, seed + 2)
    return np.vstack([o1, o2, o3]), np.vstack([d1, d2, d3])


def light_positions(g):
    dsc = g.desc().contents
    return [np.array(dsc.light_pos[3 * i:3 * i + 3]) for i in range(dsc.n_lights)]


# ---------------------------------------------------------------- comparisons
def rel_err(a, b):
    return np.abs(a - b) / np.maximum(1.0, np.abs(b))


def assert_hits_match_oracle(got, ref, what):
    """Node ids identical except at the oracle's near-ties; dist, p, normal, uv of hits within 1e-6 of max(1, |x|); misses -1,
    +inf, 0.  Returns the largest relative differences."""
    tie = ref["gap"] < TIE
    bad = (got["node"] != ref["node"]) & ~tie
    assert not bad.any(), (what, int(bad.sum()), np.argwhere(bad)[:5].ravel())
    both = (got["node"] == ref["node"]) & (ref["node"] >= 0)
    worst = {}
    for k in ("dist", "p", "normal", "uv"):
        e = rel_err(got[k][both], ref[k][both])
        worst[k] = float(e.max(initial=0))
        assert worst[k] <= 1e-6, (what, k, worst[k])
    miss = got["node"] < 0
    assert np.isposinf(got["dist"][miss]).all(), what
    for k in ("p", "normal", "uv"):
        assert (got[k][miss] == 0).all(), (what, k)
    return worst


SCENES = [("lecture4", os.path.join(SC, "lecture4.sdl")), ("lecture5", os.path.join(SC, "lecture5.sdl")),
          ("chessboard", os.path.join(SC, "chessboard.sdl")), ("zaphod", os.path.join(SC, "zaphod.sdl")),
          ("quirks", os.path.join(TSC, "quirks.sdl")), ("nested", os.path.join(TSC, "nested.sdl")),
          ("sky", os.path.join(TSC, "sky.sdl")), ("big257", None)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,path", SCENES, ids=[s[0] for s in SCENES])
def test_closest_hit_and_visibility_equal_the_oracle(ctx, orr, big_path, name, path):
    """About 50k closest-hit queries per scene (camera rays in row order, random rays in a box around the scene, rays aimed at
    node centres), then visibility from the oracle's hit points (offset by N 1e-6) to every light, and random segments.
    Measured on a B200, the largest relative differences of hits over the eight scenes: dist 2.1e-13, p 1.5e-11 (257 nodes),
    normal 5.8e-12, uv 5.6e-8 (sphere uv is FP32, render_kernel.cu local_surface)."""
    path = path or big_path
    g = c2.HostScene(path)
    if name == "big257":
        assert g.info()["nodes"] == 257
    o, d = all_queries(g)
    got, st = g.trace_rays(o, d)
    assert st.launches == 1 and st.n_gpus == 1
    ref = orr(path).trace(o, d)
    worst = assert_hits_match_oracle(got, ref, name)
    print(f"{name}: largest relative differences of hits {worst}")
    assert (got["node"] >= 0).mean() > 0.2, name

    hit = ref["node"] >= 0
    frm = ref["p"][hit] + ref["normal"][hit] * 1e-6
    lights = light_positions(g)
    rng = np.random.default_rng(7)
    lo, hi = scene_box(g)
    f = np.vstack([frm for _ in lights] + [rng.uniform(lo, hi, (N_PER_GEN, 3))])
    t = np.vstack([np.broadcast_to(L, frm.shape) for L in lights] + [rng.uniform(lo, hi, (N_PER_GEN, 3))])
    vis, _ = g.test_visibility(f, t)
    rvis, gap = orr(path).visibility(f, t)
    flagged = gap < TIE
    assert flagged.mean() <= 1e-3, (name, int(flagged.sum()))
    bad = (vis != rvis) & ~flagged
    assert not bad.any(), (name, int(bad.sum()), np.argwhere(bad)[:5].ravel())
    assert vis.any() and (~vis).any(), name


@pytest.mark.gpu
@pytest.mark.parametrize("path", [os.path.join(SC, "chessboard.sdl"), os.path.join(SC, "lecture5.sdl"), os.path.join(SC, "lecture4.sdl")])
def test_ray_to_the_pixel_picks_hit_point_reports_the_pick(ctx, path):
    g = c2.HostScene(path)
    g.set_frame_size(96, 64)
    g.override(dof=0)
    pos = camera_vectors(g)[0]
    picks = [(x, y, g.render_pixel(x, y)[1]) for y in range(0, 64, 3) for x in range(0, 96, 3)]
    picks = [(x, y, h) for x, y, h in picks if h.node >= 0]
    assert len(picks) > 100
    p = np.array([list(h.p) for _, _, h in picks])
    got, _ = g.trace_rays(np.broadcast_to(pos, p.shape), p - pos)
    want = np.array([h.node for _, _, h in picks])
    same = got["node"] == want
    assert same.mean() >= 0.995, (path, int((~same).sum()))
    dist = np.array([h.dist for _, _, h in picks])
    assert rel_err(got["dist"][same], dist[same]).max() <= 1e-6


def _bits(res):
    return {k: np.ascontiguousarray(v).view(np.uint8) for k, v in res.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["chessboard", "big257"])
def test_results_do_not_depend_on_order_or_batch(ctx, big_path, which):
    """Row order (coherent warps: the mask paths), shuffled (wide warps: the all-nodes fallback) and ragged batches give every
    query the same bits."""
    path = big_path if which == "big257" else os.path.join(SC, "chessboard.sdl")
    g = c2.HostScene(path)
    (o1, d1), (o2, d2) = all_queries(g, seed=3), all_queries(g, seed=13)
    o, d = np.vstack([o1, o2]), np.vstack([d1, d2])   # > 1 + 31 + 257 + 100003 queries
    ref, _ = g.trace_rays(o, d)
    L = light_positions(g)[0]
    hit = ref["node"] >= 0
    f = np.vstack([ref["p"][hit] + ref["normal"][hit] * 1e-6, o])
    t = np.vstack([np.broadcast_to(L, (int(hit.sum()), 3)), o + d * 3.0])
    vref, _ = g.test_visibility(f, t)
    perm = np.random.default_rng(5).permutation(len(o))
    got, _ = g.trace_rays(o[perm], d[perm])
    for k in RAY_PLANES:
        assert np.array_equal(_bits({k: got[k]})[k], _bits({k: ref[k][perm]})[k]), k
    vperm = np.random.default_rng(6).permutation(len(f))
    assert np.array_equal(g.test_visibility(f[vperm], t[vperm])[0], vref[vperm])
    start = 0
    for n in (1, 31, 257, 100003):
        part, _ = g.trace_rays(o[start:start + n], d[start:start + n])
        for k in RAY_PLANES:
            assert np.array_equal(_bits({k: part[k]})[k], _bits({k: ref[k][start:start + n]})[k]), (n, k)
        assert np.array_equal(g.test_visibility(f[start:start + n], t[start:start + n])[0], vref[start:start + n]), n
        start += n


@pytest.mark.gpu
def test_global_memory_form_gives_the_same_bits(ctx, monkeypatch):
    path = os.path.join(SC, "lecture5.sdl")
    g = c2.HostScene(path)
    o, d = all_queries(g, seed=9)
    const, _ = g.trace_rays(o, d)
    vc, _ = g.test_visibility(o, o + d)
    monkeypatch.setenv("C2RT_FORCE_GLOBAL", "1")   # read at scene-create time
    g2 = c2.HostScene(path)
    glob, _ = g2.trace_rays(o, d)
    vg, _ = g2.test_visibility(o, o + d)
    for k in RAY_PLANES:
        assert np.array_equal(_bits(const)[k], _bits(glob)[k]), k
    assert np.array_equal(vc, vg)


@pytest.mark.gpu
def test_device_entry_points_on_a_side_stream_with_guard_words(ctx):
    import torch
    g = c2.HostScene(os.path.join(SC, "chessboard.sdl"))
    o, d = all_queries(g, seed=4)
    n = len(o) - 5   # a ragged tail
    o, d = o[:n], d[:n]
    ref, _ = g.trace_rays(o, d)
    vref, _ = g.test_visibility(o, o + d)
    handle = g.device_scene()
    stream = torch.cuda.Stream()
    guard = 64
    with torch.cuda.stream(stream):
        to, td, tt = (torch.from_numpy(a).to("cuda") for a in (o, d, o + d))
        bufs = {k: torch.full((n * max(1, s) + 2 * guard,), 7.0 if k != "node" else 7,
                              dtype=torch.int32 if k == "node" else torch.float64, device="cuda")
                for k, s in (("node", 1), ("dist", 1), ("p", 3), ("normal", 3), ("uv", 2))}
        vis = torch.full((n + 2 * guard,), 0x5A, dtype=torch.uint8, device="cuda")
    esz = {k: b.element_size() for k, b in bufs.items()}
    api.trace_rays_device(handle, n, to.data_ptr(), td.data_ptr(), *(bufs[k].data_ptr() + guard * esz[k] for k in RAY_PLANES),
                          stream=stream.cuda_stream)
    api.test_visibility_device(handle, n, to.data_ptr(), tt.data_ptr(), vis.data_ptr() + guard, stream=stream.cuda_stream)
    stream.synchronize()
    for k in RAY_PLANES:
        b = bufs[k].cpu().numpy()
        assert (b[:guard] == 7).all() and (b[-guard:] == 7).all(), k
        assert np.array_equal(b[guard:-guard].view(np.uint8), np.ascontiguousarray(ref[k]).reshape(-1).view(np.uint8)), k
    v = vis.cpu().numpy()
    assert (v[:guard] == 0x5A).all() and (v[-guard:] == 0x5A).all()
    assert np.array_equal(v[guard:-guard].astype(bool), vref)


@pytest.mark.gpu
def test_two_devices_give_the_one_device_bits():
    if c2.device_count() < 2:
        pytest.skip("needs two GPUs")
    path = os.path.join(SC, "chessboard.sdl")
    c2.init(1, [0])
    try:
        g = c2.HostScene(path)
        o, d = all_queries(g)
        one, _ = g.trace_rays(o, d)
        v1, _ = g.test_visibility(o, o + d)
        c2.init(2)
        g = c2.HostScene(path)
        two, st = g.trace_rays(o, d)
        v2, _ = g.test_visibility(o, o + d)
        assert st.n_gpus == 2 and st.launches == 2
        for k in RAY_PLANES:
            assert np.array_equal(_bits(one)[k], _bits(two)[k]), k
        assert np.array_equal(v1, v2)
    finally:
        c2.shutdown()


@pytest.mark.gpu
def test_untraced_queries_and_origins_on_surfaces(ctx, orr):
    """A zero direction, NaN or infinite coordinates and from == to are not traced: a miss, visible = 1.  Origins inside a
    sphere and on the floor plane are traced like any other query, as the oracle does."""
    path = os.path.join(SC, "lecture5.sdl")
    g = c2.HostScene(path)
    nan, inf = float("nan"), float("inf")
    o = np.array([[0, 5, 0], [nan, 5, 0], [0, 5, 0], [inf, 5, 0], [0, 5, 0], [0, 5, 0], [0, 5, 0]], np.float64)
    d = np.array([[0, 0, 0], [0, -1, 0], [0, nan, 0], [0, -1, 0], [-inf, -1, 0], [1e-200, 0, 0], [0, 1e300, 0]], np.float64)
    got, _ = g.trace_rays(o, d)
    assert (got["node"] == -1).all() and np.isposinf(got["dist"]).all()
    for k in ("p", "normal", "uv"):
        assert (got[k] == 0).all(), k
    vis, _ = g.test_visibility(np.vstack([o, [[0, 5, 0]]]), np.vstack([o + d, [[0, 5, 0]]]))
    assert vis.all()
    # origins inside the sphere nodes and exactly on the floor (y = the plane's height), compared with the oracle
    cen = node_centres(g)
    rng = np.random.default_rng(2)
    oi = np.repeat(cen, 50, axis=0) + rng.normal(scale=1e-3, size=(len(cen) * 50, 3))
    floor = np.column_stack([rng.uniform(-50, 50, 200), np.zeros(200), rng.uniform(-50, 50, 200)])
    oq = np.vstack([oi, floor])
    dq = rng.normal(size=oq.shape)
    got, _ = g.trace_rays(oq, dq)
    assert_hits_match_oracle(got, orr(path).trace(oq, dq), "origins on surfaces")
    t = oq + dq * 40
    vis, _ = g.test_visibility(oq, t)
    rvis, gap = orr(path).visibility(oq, t)
    ok = gap >= TIE
    assert np.array_equal(vis[ok], rvis[ok])


@pytest.mark.gpu
def test_queries_leave_colour_frames_counters_and_cancel_alone(ctx):
    g = c2.HostScene(os.path.join(SC, "lecture5.sdl"))
    g.set_frame_size(97, 61)
    before, argb0, st0 = g.render(argb=True, count_rays=True)
    handle = g.device_scene()
    assert api.read_ray_counters(handle) == (0, 0)
    o, d = all_queries(g)
    r1, _ = g.trace_rays(o, d)
    v1, _ = g.test_visibility(o, o + d)
    assert api.read_ray_counters(handle) == (0, 0)
    api.cancel()   # no frame in progress: cancels nothing, and a query neither takes nor leaves the request
    r2, _ = g.trace_rays(o, d)
    v2, _ = g.test_visibility(o, o + d)
    after, argb1, st1 = g.render(argb=True, count_rays=True)
    assert not g.cancelled
    assert np.array_equal(before.view(np.uint32), after.view(np.uint32)) and np.array_equal(argb0, argb1)
    assert (st0.primary_rays, st0.shadow_rays) == (st1.primary_rays, st1.shadow_rays)
    for k in RAY_PLANES:
        assert np.array_equal(_bits(r1)[k], _bits(r2)[k]), k
    assert np.array_equal(v1, v2)


@pytest.mark.gpu
def test_queries_interleaved_with_colour_frames_of_another_scene(ctx):
    a = c2.HostScene(os.path.join(SC, "chessboard.sdl"))
    b = c2.HostScene(os.path.join(SC, "lecture5.sdl"))
    b.set_frame_size(64, 48)
    o, d = all_queries(a, seed=12)
    ref, _ = a.trace_rays(o, d)
    vref, _ = a.test_visibility(o, o + d)
    frame0, _, _ = b.render()
    for _ in range(2):
        got, _ = a.trace_rays(o, d)
        frame, _, _ = b.render()
        vis, _ = a.test_visibility(o, o + d)
        for k in RAY_PLANES:
            assert np.array_equal(_bits(got)[k], _bits(ref)[k]), k
        assert np.array_equal(vis, vref)
        assert np.array_equal(frame.view(np.uint32), frame0.view(np.uint32))


# ---------------------------------------------------------------- no GPU needed
BOGUS = C.c_void_p(16)   # never dereferenced: the argument checks come first


def test_argument_errors_come_before_any_device():
    o = np.zeros((4, 3))
    node = np.zeros(4, np.int32)
    out = api.RayHits(node.ctypes.data, None, None, None, None)
    none = api.RayHits()
    vis = np.zeros(4, np.uint8)
    L = api.lib
    assert L.c2rt_trace_rays(None, 4, o.ctypes.data, o.ctypes.data, C.byref(out), None) == -1
    assert L.c2rt_trace_rays(BOGUS, 4, None, o.ctypes.data, C.byref(out), None) == -1
    assert L.c2rt_trace_rays(BOGUS, 4, o.ctypes.data, None, C.byref(out), None) == -1
    assert L.c2rt_trace_rays(BOGUS, 4, o.ctypes.data, o.ctypes.data, C.byref(none), None) == -1
    assert "output is null" in L.c2rt_last_error().decode()
    assert L.c2rt_trace_rays(BOGUS, 4, o.ctypes.data, o.ctypes.data, None, None) == -1
    assert L.c2rt_trace_rays_device(BOGUS, 4, None, o.ctypes.data, C.byref(out), None, None) == -1
    assert L.c2rt_trace_rays_device(BOGUS, 4, o.ctypes.data, o.ctypes.data, C.byref(none), None, None) == -1
    assert L.c2rt_test_visibility(BOGUS, 4, o.ctypes.data, None, vis.ctypes.data, None) == -1
    assert L.c2rt_test_visibility(BOGUS, 4, o.ctypes.data, o.ctypes.data, None, None) == -1
    assert L.c2rt_test_visibility_device(None, 4, o.ctypes.data, o.ctypes.data, vis.ctypes.data, None, None) == -1
    assert L.c2rt_test_visibility_device(BOGUS, 4, o.ctypes.data, o.ctypes.data, None, None, None) == -1
    big = 2 ** 31
    assert L.c2rt_trace_rays(BOGUS, big, o.ctypes.data, o.ctypes.data, C.byref(out), None) == -5
    assert L.c2rt_trace_rays_device(BOGUS, big, o.ctypes.data, o.ctypes.data, C.byref(out), None, None) == -5
    assert L.c2rt_test_visibility(BOGUS, big, o.ctypes.data, o.ctypes.data, vis.ctypes.data, None) == -5
    assert L.c2rt_test_visibility_device(BOGUS, big, o.ctypes.data, o.ctypes.data, vis.ctypes.data, None, None) == -5
    # n == 0: a no-op (the inputs may then be null), stats zeroed
    st = api.Stats(kernel_ms=5.0, launches=9)
    assert L.c2rt_trace_rays(BOGUS, 0, None, None, C.byref(out), C.byref(st)) == 0
    assert (st.kernel_ms, st.launches) == (0.0, 0)
    assert L.c2rt_test_visibility_device(BOGUS, 0, None, None, vis.ctypes.data, None, None) == 0


@pytest.mark.skipif(HAS_GPU, reason="checks the failure without a GPU")
def test_without_a_gpu_valid_queries_fail_with_a_cuda_error():
    o = np.zeros((4, 3))
    d = np.ones((4, 3))
    vis = np.zeros(4, np.uint8)
    node = np.zeros(4, np.int32)
    out = api.RayHits(node.ctypes.data, None, None, None, None)
    assert api.lib.c2rt_trace_rays(BOGUS, 4, o.ctypes.data, d.ctypes.data, C.byref(out), None) == -3
    assert api.lib.c2rt_test_visibility(BOGUS, 4, o.ctypes.data, d.ctypes.data, vis.ctypes.data, None) == -3
    g = c2.HostScene(os.path.join(SC, "lecture4.sdl"))
    for call in (lambda: g.trace_rays(o, d), lambda: g.test_visibility(o, d)):
        with pytest.raises(c2.C2rtError) as e:
            call()
        assert e.value.status == -3


def test_ray_query_bindings_follow_the_header():
    header = open(os.path.join(ROOT, "include", "c2rt.h")).read()
    assert "typedef struct c2rt_ray_hits" in header
    body = header.split("typedef struct c2rt_ray_hits")[1].split("} c2rt_ray_hits;")[0]
    fields = [line.split("*")[1].split(";")[0].strip() for line in body.splitlines()[1:] if ";" in line and "*" in line]
    assert fields == [f[0] for f in api.RayHits._fields_] == list(api.RAY_PLANES) == list(RAY_PLANES)
    assert C.sizeof(api.RayHits) == 5 * 8
    names = {"c2rt_trace_rays", "c2rt_trace_rays_device", "c2rt_test_visibility", "c2rt_test_visibility_device"}
    assert names <= set(api.C_ABI_SYMBOLS)
    for n in names:
        assert f"int {n}(" in header, n
    g = c2.HostScene(os.path.join(SC, "lecture4.sdl"))
    with pytest.raises(ValueError):
        g.trace_rays(np.zeros((3, 3)), np.zeros((2, 3)))
    with pytest.raises(ValueError):
        g.trace_rays(np.zeros((3, 3)), np.zeros((3, 3)), planes=("depth",))
    with pytest.raises(ValueError):
        g.test_visibility(np.zeros((3, 2)), np.zeros((3, 2)))
