"""Node edits in place (c2rt_scene_set_nodes, HostScene.place_node): after an edit every call on the uploaded scene gives the
bits of a scene created fresh from the edited scene file — colour frames (RGB and ARGB), hit frames, the pixel pick, ray
queries, visibility and shaded rays — across scene classes, the global-memory form, residency changes, the device route, a
frame running on another thread, and two devices."""
import ctypes as C
import os
import threading
import time

import numpy as np
import pytest

import chess2rt_b200 as c2
from chess2rt_b200 import api
from sdl_edit import SC, TSC, edit_node, load_edited, write_scene

HAS_GPU = c2.device_count() > 0
SIZE = (160, 90)
CHESS = os.path.join(SC, "chessboard.sdl")
LECTURE5 = os.path.join(SC, "lecture5.sdl")
PROC = os.path.join(SC, "lecture4-proc-texture.sdl")
ZAPHOD = os.path.join(SC, "zaphod.sdl")
NESTED = os.path.join(TSC, "nested.sdl")


@pytest.fixture(scope="module")
def ctx():
    c2.init(1, [0])
    yield
    c2.shutdown()


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def ray_set(handle_scene, n=3000, seed=5):
    """A fixed set of queries around the scene's camera: origins near it, directions into the lower half-space, visibility
    segments from the origins to points on and above y = 0."""
    cam, _ = handle_scene.frame_blocks()
    rng = np.random.default_rng(seed)
    o = np.array(list(cam.pos)) + rng.normal(0.0, 5.0, (n, 3))
    d = rng.normal(0.0, 1.0, (n, 3))
    d[:, 1] = -np.abs(d[:, 1]) - 0.3
    to = np.array(list(cam.pos)) * [1, 0, 1] + rng.normal(0.0, 60.0, (n, 3)) * [1, 0, 1] + rng.uniform(0, 30, (n, 1)) * [0, 1, 0]
    return o, d, to


def outputs(handle, cam, st, ambient, rays):
    """Everything a host can ask of an uploaded scene, raw bits: colour frame (rgb, argb), hit frame, a few pixel picks,
    closest hits, visibility and shaded rays of `rays`."""
    w, h = st.frame_width, st.frame_height
    out = {}
    rgb, argb = np.empty((h, w, 3), np.float32), np.empty((h, w), np.uint32)
    assert api.lib.c2rt_render(handle, C.byref(cam), C.byref(st), rgb.ctypes.data, argb.ctypes.data, None) == 0, api.lib.c2rt_last_error()
    out["rgb"], out["argb"] = bits(rgb), argb
    planes = {k: np.empty((h, w) + shape, dt) for k, (dt, shape) in api.HIT_PLANES.items()}
    p = api.HitPlanes(*(planes[k].ctypes.data for k in api.HIT_PLANES))
    assert api.lib.c2rt_render_hits(handle, C.byref(cam), C.byref(st), C.byref(p), None) == 0, api.lib.c2rt_last_error()
    out.update({"hit_" + k: bits(v) for k, v in planes.items()})
    pix, hit = (C.c_float * 3)(), api.Hit()
    picks = []
    for x, y in ((0, 0), (w // 2, h // 2), (w // 3, 2 * h // 3), (w - 1, h - 1), (3 * w // 4, h // 4)):
        if api.lib.c2rt_render_pixel(handle, C.byref(cam), C.byref(st), x, y, pix, C.byref(hit)) == 0:
            picks.append(bytes(pix) + bytes(hit))
        else:   # GI / refused frames: the refusal is the output
            picks.append(api.lib.c2rt_last_error())
    out["picks"] = picks
    o, d, to = rays
    n = len(o)
    rp = {k: np.empty((n,) + shape, dt) for k, (dt, shape) in api.RAY_PLANES.items()}
    rh = api.RayHits(*(rp[k].ctypes.data for k in api.RAY_PLANES))
    assert api.lib.c2rt_trace_rays(handle, n, o.ctypes.data, d.ctypes.data, C.byref(rh), None) == 0
    out.update({"ray_" + k: v.view(np.uint8) for k, v in rp.items()})
    vis = np.empty(n, np.uint8)
    assert api.lib.c2rt_test_visibility(handle, n, o.ctypes.data, to.ctypes.data, vis.ctypes.data, None) == 0
    out["visible"] = vis
    srgb, sargb = np.empty((n, 3), np.float32), np.empty(n, np.uint32)
    amb = (C.c_float * 3)(*ambient)
    assert api.lib.c2rt_shade_rays(handle, amb, n, o.ctypes.data, d.ctypes.data, srgb.ctypes.data, sargb.ctypes.data, None) == 0
    out["shade_rgb"], out["shade_argb"] = bits(srgb), sargb
    return out


def scene_outputs(s, rays, seed=3):
    cam, st = s.frame_blocks(seed=seed)
    return outputs(s.device_scene(), cam, st, st.ambient_light, rays)


def assert_same(a, b, what=""):
    assert a.keys() == b.keys()
    for k in a:
        if k == "picks":
            assert a[k] == b[k], (what, k)
        else:
            assert np.array_equal(a[k], b[k]), (what, k, int((a[k] != b[k]).sum()))


def load(path, size=SIZE):
    s = c2.HostScene(path)
    s.set_frame_size(*size)
    return s


# (id, scene, [(node, place_node keywords)]): chess move / capture / promotion; lecture5's globe leaves the world-space sphere
# path (the rotate key scales, as in the reference); the one-plane scene keeps its diagonal plane (MODE_SOLO); zaphod with DOF
EDITS = [
    ("chess_move", CHESS, [("e2", dict(translate=(10.0, 0.0, -10.0)))]),
    ("chess_capture", CHESS, [("d7", dict(translate=(130.0, 0.0, 40.0)))]),
    ("chess_promotion", CHESS, [("a7", dict(geometry="queen", translate=(-70.0, 0.0, 70.0)))]),
    ("chess_many", CHESS, [("e2", dict(translate=(10.0, 0.0, -10.0))), ("e7", dict(translate=(10.0, 0.0, 10.0))),
                           ("g1", dict(translate=(10.0, 0.0, -50.0))), ("c1", dict(translate=(-30.0, 0.0, -70.0)))]),
    ("lecture5_globe_generic", LECTURE5, [("globe", dict(rotate=(1.5, 0.5, 2.0)))]),
    ("lecture5_csg_and_ball", LECTURE5, [("csgNode", dict(translate=(-20.0, 5.0, 30.0))), ("S3", dict(geometry="globe_ball"))]),
    ("proc_plane_solo", PROC, [("floor", dict(scale=(2.0, 1.0, 0.5), translate=(3.0, -4.0, 7.0)))]),
    ("zaphod_dof", ZAPHOD, [("book", dict(scale=(10.0, 10.0, 10.0), translate=(0.5, -1.0, 2.0)))]),
    ("nested", NESTED, [("c", dict(translate=(0.0, 30.0, 20.0))), ("d", dict(geometry="deeper", translate=(70.0, 20.0, -20.0)))]),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,path,edits", EDITS, ids=[e[0] for e in EDITS])
def test_edit_gives_the_fresh_scene_bits(ctx, tmp_path, name, path, edits):
    s = load(path)
    rays = ray_set(s)
    before = scene_outputs(s, rays)   # uploaded and resident before the edit
    for node, kw in edits:
        s.place_node(node, **kw)
    after = scene_outputs(s, rays)
    fresh = load_edited(str(tmp_path), path, edits)
    fresh.set_frame_size(*SIZE)
    assert_same(after, scene_outputs(fresh, rays), name)
    assert any(not np.array_equal(before[k], after[k]) for k in ("rgb", "hit_node", "ray_dist")), "the edit changed nothing"


@pytest.mark.gpu
def test_global_memory_form(ctx, tmp_path, monkeypatch):
    monkeypatch.setenv("C2RT_FORCE_GLOBAL", "1")   # read at scene-create time, by both scenes
    edits = [("a7", dict(geometry="queen", translate=(-70.0, 0.0, 70.0))), ("d7", dict(translate=(130.0, 0.0, 40.0)))]
    s = load(CHESS)
    rays = ray_set(s)
    scene_outputs(s, rays)
    for node, kw in edits:
        s.place_node(node, **kw)
    fresh = load_edited(str(tmp_path), CHESS, edits)
    fresh.set_frame_size(*SIZE)
    assert_same(scene_outputs(s, rays), scene_outputs(fresh, rays))


def rotation_y(deg):
    a = np.radians(deg)
    return np.array([[np.cos(a), 0, -np.sin(a)], [0, 1, 0], [np.sin(a), 0, np.cos(a)]])


def edited_desc_scene(s, node, m, off):
    """A scene created by c2rt_scene_create from `s`'s flat description with node `node`'s transform replaced (the
    description is edited in place, as a host holding the arrays would)."""
    d = s.desc()
    dc = d.contents
    inv = np.linalg.inv(m)
    for arr, v in ((dc.node_transform, m), (dc.node_inverse, inv), (dc.node_inverse_t, inv.T)):
        for k in range(9):
            arr[9 * node + k] = float(v.reshape(-1)[k])
    for k in range(3):
        dc.node_offset[3 * node + k] = float(off[k])
    h = C.c_void_p()
    assert api.lib.c2rt_scene_create(d, C.byref(h)) == 0, api.lib.c2rt_last_error()
    return h


@pytest.mark.gpu
@pytest.mark.parametrize("path,node,deg,off", [(LECTURE5, "globe", 30.0, (5.0, 2.0, -3.0)), (LECTURE5, "floor", 0.0, (0.0, -2.0, 0.0)),
                                               (PROC, "floor", 20.0, (0.0, 1.0, 0.0)), (PROC, "floor", 0.0, (4.0, -3.0, 2.0))],
                         ids=["lecture5_globe_rotated", "lecture5_floor_lowered", "proc_plane_rotated_leaves_solo", "proc_plane_moved_stays_solo"])
def test_raw_transforms_give_the_fresh_scene_bits(ctx, path, node, deg, off):
    """c2rt_scene_set_nodes with true rotations (which the scene format cannot express): a rotated world-space sphere becomes a
    generic node, a rotated one-plane scene leaves MODE_SOLO, a moved one stays."""
    s = load(path)
    rays = ray_set(s)
    scene_outputs(s, rays)
    i = s.node_index(node)
    m = rotation_y(deg)
    inv = np.linalg.inv(m)
    c2.scene_set_nodes(s.device_scene(), [i], transform=m, inverse=inv, inverse_t=inv.T, offset=off)
    after = scene_outputs(s, rays)
    ref = load(path)
    h = edited_desc_scene(ref, i, m, off)
    try:
        cam, st = ref.frame_blocks(seed=3)
        assert_same(after, outputs(h, cam, st, st.ambient_light, rays))
    finally:
        api.lib.c2rt_scene_destroy(h)


@pytest.mark.gpu
def test_edit_then_undo_gives_the_original_bits(ctx):
    for path, node, there, back in ((CHESS, "e2", dict(geometry="queen", translate=(10.0, 0.0, -10.0)), dict(geometry="pawn", translate=(10.0, 0.0, -50.0))),
                                    (PROC, "floor", dict(scale=(1.0, 1.0, 2.0)), dict())):
        s = load(path)
        rays = ray_set(s)
        orig = scene_outputs(s, rays)
        s.place_node(node, **there)
        scene_outputs(s, rays)
        s.place_node(node, **back)
        assert_same(scene_outputs(s, rays), orig, path)


@pytest.mark.gpu
def test_a_refused_edit_changes_no_output(ctx):
    s = load(CHESS)
    rays = ray_set(s)
    orig = scene_outputs(s, rays)
    h = s.device_scene()
    n_nodes, n_geoms = s.info()["nodes"], s.info()["geometries"]
    m = np.eye(3)
    bad = [dict(nodes=[1, n_nodes], geom=[0, 0]),                      # a node index out of range (after a valid entry)
           dict(nodes=[1], geom=[n_geoms]), dict(nodes=[1], geom=[-1]),   # geometry indices out of range
           dict(nodes=[1], transform=m, inverse=m, offset=(0, 0, 0)),     # a partial set of transform arrays
           dict(nodes=[1])]                                               # nothing to edit
    for kw in bad:
        with pytest.raises(c2.C2rtError) as e:
            c2.scene_set_nodes(h, **kw)
        assert e.value.status == -1, kw
    rc = api.lib.c2rt_scene_set_nodes(h, 1, None, np.zeros(1, np.int32).ctypes.data, None, None, None, None)
    assert rc == -1 and b"nodes is null" in api.lib.c2rt_last_error()
    c2.scene_set_nodes(h, [], geom=[])   # n == 0: a no-op
    with pytest.raises(c2.C2rtError):
        s.place_node("a2", geometry="dragon", translate=(0, 0, 0))
    assert_same(scene_outputs(s, rays), orig)


@pytest.mark.gpu
def test_later_entries_for_the_same_node_win(ctx, tmp_path):
    s = load(CHESS)
    rays = ray_set(s)
    i = s.node_index("e2")
    q = s.node_index("d1")
    d = s.desc().contents
    queen = d.node_geom[q]
    c2.scene_set_nodes(s.device_scene(), [i, i], geom=[0, queen])
    fresh = load_edited(str(tmp_path), CHESS, [("e2", dict(geometry="queen", translate=(10.0, 0.0, -50.0)))])
    fresh.set_frame_size(*SIZE)
    assert_same(outputs(s.device_scene(), *s.frame_blocks(seed=3)[:2], (0.0, 0.0, 0.0), rays),
                outputs(fresh.device_scene(), *fresh.frame_blocks(seed=3)[:2], (0.0, 0.0, 0.0), rays))


@pytest.mark.gpu
def test_edit_while_another_scene_is_resident(ctx, tmp_path):
    edits = [("e2", dict(translate=(10.0, 0.0, -10.0)))]
    a, b = load(CHESS), load(LECTURE5)
    rays_a, rays_b = ray_set(a), ray_set(b)
    scene_outputs(a, rays_a)
    b_before = scene_outputs(b, rays_b)   # b is now the resident scene
    for node, kw in edits:
        a.place_node(node, **kw)
    assert_same(scene_outputs(b, rays_b), b_before)
    fresh = load_edited(str(tmp_path), CHESS, edits)
    fresh.set_frame_size(*SIZE)
    assert_same(scene_outputs(a, rays_a), scene_outputs(fresh, rays_a))


@pytest.mark.gpu
def test_device_route_after_an_edit_matches_the_host_route(ctx):
    import torch
    s = load(CHESS, (192, 108))
    h = s.device_scene()
    stream = torch.cuda.Stream()
    w, hh = s.frame_size
    d_rgb = torch.empty(hh * w * 3, dtype=torch.float32, device="cuda")
    d_argb = torch.empty(hh * w, dtype=torch.int32, device="cuda")
    cam, st = s.frame_blocks(seed=1)
    api.render_device(h, cam, st, d_rgb.data_ptr(), d_argb.data_ptr(), stream=stream.cuda_stream)   # resident on the stream
    stream.synchronize()
    s.place_node("a7", geometry="queen", translate=(-70.0, 0.0, 70.0))
    cam, st = s.frame_blocks(seed=1)
    api.render_device(h, cam, st, d_rgb.data_ptr(), d_argb.data_ptr(), stream=stream.cuda_stream)
    stream.synchronize()
    rgb, argb, _ = s.render(argb=True, seed=1)
    assert np.array_equal(bits(d_rgb.cpu().numpy()), bits(rgb.reshape(-1)))
    assert np.array_equal(d_argb.cpu().numpy().view(np.uint32), argb.reshape(-1))


@pytest.mark.gpu
def test_an_edit_waits_for_a_frame_on_another_thread(ctx, tmp_path):
    """The edit takes the library lock: a frame running on another thread completes as the pre-edit or the post-edit frame,
    never a mixture."""
    size = (1920, 1080)
    edits = [("a7", dict(geometry="queen", translate=(-70.0, 0.0, 70.0))), ("e2", dict(translate=(10.0, 0.0, -10.0)))]
    s = load(CHESS, size)
    post_scene = load_edited(str(tmp_path), CHESS, edits)
    post_scene.set_frame_size(*size)
    post_desc = post_scene.desc().contents
    idx = [s.node_index(n) for n, _ in edits]
    arr = lambda p, per: np.array([[p[per * i + k] for k in range(per)] for i in idx])  # noqa: E731
    geom = [post_desc.node_geom[i] for i in idx]
    tf = [arr(post_desc.node_transform, 9), arr(post_desc.node_inverse, 9), arr(post_desc.node_inverse_t, 9), arr(post_desc.node_offset, 3)]
    cam, st = s.frame_blocks(seed=2)
    h = s.device_scene()

    def frame():
        rgb = np.empty((size[1], size[0], 3), np.float32)
        assert api.lib.c2rt_render(h, C.byref(cam), C.byref(st), rgb.ctypes.data, None, None) == 0
        return bits(rgb)

    pre = frame()
    frames, started = [], threading.Event()

    def worker():
        started.set()
        for _ in range(12):
            frames.append(frame())

    t = threading.Thread(target=worker)
    t.start()
    started.wait()
    time.sleep(0.002)
    c2.scene_set_nodes(h, idx, geom=geom, transform=tf[0], inverse=tf[1], inverse_t=tf[2], offset=tf[3])
    t.join()
    assert len(frames) == 12
    post_rgb, _, _ = post_scene.render(seed=2)
    post = bits(post_rgb)
    assert not np.array_equal(pre, post)
    for k, f in enumerate(frames):
        assert np.array_equal(f, pre) or np.array_equal(f, post), k
    assert np.array_equal(frame(), post)


@pytest.mark.gpu
def test_oracle_parity_of_an_edited_chessboard(ctx, tmp_path):
    from oracle_binding import OracleScene, parity_report
    edits = [("a7", dict(geometry="queen", translate=(-70.0, 0.0, 70.0))), ("d7", dict(translate=(130.0, 0.0, 40.0))),
             ("e2", dict(translate=(10.0, 0.0, -10.0)))]
    s = load(CHESS, (240, 135))
    s.render()
    for node, kw in edits:
        s.place_node(node, **kw)
    rgb, argb, _ = s.render(argb=True)
    with open(CHESS) as fh:
        text = fh.read()
    for node, kw in edits:
        text = edit_node(text, node, **kw)
    o = OracleScene(write_scene(str(tmp_path), CHESS, text))
    o.set_frame_size(240, 135)
    ref, _ = o.render()
    rep = parity_report(rgb, ref, argb)
    assert rep["px_over_1e-3"] == 0 and rep["frac_over_1lsb"] <= 1e-3, rep


@pytest.mark.gpu
@pytest.mark.skipif(c2.device_count() < 2, reason="needs two GPUs")
def test_two_devices_give_the_fresh_scene_bits(tmp_path):
    edits = [("a7", dict(geometry="queen", translate=(-70.0, 0.0, 70.0))), ("d7", dict(translate=(130.0, 0.0, 40.0)))]
    c2.init(2, [0, 1])
    try:
        s = load(CHESS, (320, 180))
        rays = ray_set(s, n=9000)
        scene_outputs(s, rays)
        for node, kw in edits:
            s.place_node(node, **kw)
        fresh = load_edited(str(tmp_path), CHESS, edits)
        fresh.set_frame_size(320, 180)
        assert_same(scene_outputs(s, rays), scene_outputs(fresh, rays))
    finally:
        c2.init(1, [0])
