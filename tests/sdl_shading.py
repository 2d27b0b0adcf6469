"""Shading and light edits written into scene text: the scene file a host would have loaded after re-shading, re-texturing or
relighting.  The shading-edit tests compare HostScene.set_* / c2rt_scene_set_* against a scene loaded fresh from that text;
this module also holds the output bundle they compare (every call a host can make on an uploaded scene)."""
import ctypes as C
import re

import numpy as np

import chess2rt_b200 as c2
from chess2rt_b200 import api
from sdl_edit import write_scene


def _match_brace(text, i):
    """The index just past the `}` closing the block whose body starts at i."""
    depth = 1
    while depth:
        depth += {"{": 1, "}": -1}.get(text[i], 0)
        i += 1
    return i


def _section(text, section):
    """(start, end) of the body of the scene's `section { ... }` block (Lights, Textures, Shaders, Nodes)."""
    m = re.search(r"\b%s\s*\{" % section, text)
    if not m:
        raise KeyError(section)
    return m.end(), _match_brace(text, m.end()) - 1


def _statements(body):
    """The top-level statements of a block body: one per line or `;`, a `key { ... }` sub-block as one statement."""
    out, i, n = [], 0, len(body)
    while i < n:
        j = body.find("\n", i)
        j = n if j < 0 else j
        line = body[i:j]
        if "{" in line:
            k = _match_brace(body, i + line.index("{") + 1)
            out.append(body[i:k].strip())
            i = k
            continue
        out += [s.strip() for s in line.split("//")[0].split(";") if s.strip()]
        i = j + 1
    return out


def _entities(text, section):
    """(header start, body start, body end, type, name) of every entity block of a section."""
    start, end = _section(text, section)
    out = []
    for m in re.finditer(r'\b([A-Za-z0-9]+)\s*("([^"]*)")?\s*\{', text[start:end]):
        b0 = start + m.end()
        b1 = _match_brace(text, b0) - 1
        if any(b0 > e0 and b1 < e1 for _, e0, e1, _, _ in out):
            continue   # a sub-block (colorU { ... }) of an entity already listed
        name = m.group(3)
        if name is None:
            nm = re.search(r'^\s*name\s+"([^"]*)"', text[b0:b1], re.M)
            name = nm.group(1) if nm else None
        out.append((start + m.start(), b0, b1, m.group(1), name))
    return out


def _value(key, v):
    if isinstance(v, str):
        return '%s "%s"' % (key, v)
    a = np.asarray(v, np.float64)
    if a.ndim == 2:   # Procedure2 colorU / colorV: a sub-block of three colours
        return "%s {\n%s\n      }" % (key, "\n".join("        color " + " ".join(repr(float(x)) for x in c) for c in a))
    return "%s %s" % (key, " ".join(repr(float(x)) for x in a.reshape(-1)))


def edit_entity(text, section, entity, kind=None, **keys):
    """`text` with the entity named `entity` of `section` edited: kind (a block type) replaces the block's type and drops every key
    but its name, as a fresh object of that kind; each key=value replaces (or adds) that key; key=None drops it."""
    for h0, b0, b1, typ, name in _entities(text, section):
        if name != entity:
            continue
        stmts = _statements(text[b0:b1])
        if kind is not None:
            stmts = [s for s in stmts if s.split()[0] == "name"]
        stmts = [s for s in stmts if s.split()[0] not in keys]
        stmts += [_value(k, v) for k, v in keys.items() if v is not None]
        header = text[h0:b0]
        if kind is not None:
            header = kind + header[len(typ):]
        return text[:h0] + header + "\n      " + "\n      ".join(stmts) + "\n    " + text[b1:]
    raise KeyError((section, entity))


def add_entity(text, section, block):
    """`text` with `block` (an entity's whole text) appended to `section`."""
    _, end = _section(text, section)
    return text[:end] + "  " + block + "\n  " + text[end:]


def load_text(tmp_dir, src_path, text, size=None):
    s = c2.HostScene(write_scene(tmp_dir, src_path, text))
    if size:
        s.set_frame_size(*size)
    return s


def read(path):
    with open(path) as fh:
        return fh.read()


# ---------------------------------------------------------------- the output bundle of an uploaded scene

def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def ray_set(scene, n=3000, seed=5):
    """A fixed set of queries around the scene's camera: origins near it, directions into the lower half-space, visibility
    segments from the origins to points on and above y = 0."""
    cam, _ = scene.frame_blocks()
    rng = np.random.default_rng(seed)
    o = np.array(list(cam.pos)) + rng.normal(0.0, 5.0, (n, 3))
    d = rng.normal(0.0, 1.0, (n, 3))
    d[:, 1] = -np.abs(d[:, 1]) - 0.3
    to = np.array(list(cam.pos)) * [1, 0, 1] + rng.normal(0.0, 60.0, (n, 3)) * [1, 0, 1] + rng.uniform(0, 30, (n, 1)) * [0, 1, 0]
    return o, d, to


def outputs(handle, cam, st, ambient, rays):
    """Everything a host can ask of an uploaded scene, raw bits: colour frame (rgb, argb), hit frame, a few pixel picks,
    closest hits, visibility and shaded rays of `rays`.  A refused frame or pick (GI) records the refusal instead."""
    w, h = st.frame_width, st.frame_height
    out = {}
    rgb, argb = np.empty((h, w, 3), np.float32), np.empty((h, w), np.uint32)
    rc = api.lib.c2rt_render(handle, C.byref(cam), C.byref(st), rgb.ctypes.data, argb.ctypes.data, None)
    if rc == 0:
        out["rgb"], out["argb"] = bits(rgb), argb
    else:
        out["frame_refused"] = (rc, api.lib.c2rt_last_error())
    planes = {k: np.empty((h, w) + shape, dt) for k, (dt, shape) in api.HIT_PLANES.items()}
    p = api.HitPlanes(*(planes[k].ctypes.data for k in api.HIT_PLANES))
    rc = api.lib.c2rt_render_hits(handle, C.byref(cam), C.byref(st), C.byref(p), None)
    if rc == 0:
        out.update({"hit_" + k: bits(v) for k, v in planes.items()})
    else:
        out["hits_refused"] = (rc, api.lib.c2rt_last_error())
    pix, hit = (C.c_float * 3)(), api.Hit()
    picks = []
    for x, y in ((0, 0), (w // 2, h // 2), (w // 3, 2 * h // 3), (w - 1, h - 1), (3 * w // 4, h // 4)):
        if api.lib.c2rt_render_pixel(handle, C.byref(cam), C.byref(st), x, y, pix, C.byref(hit)) == 0:
            picks.append(bytes(pix) + bytes(hit))
        else:
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
    assert a.keys() == b.keys(), (what, a.keys() ^ b.keys())
    for k in a:
        if isinstance(a[k], np.ndarray):
            assert np.array_equal(a[k], b[k]), (what, k, int((a[k] != b[k]).sum()))
        else:
            assert a[k] == b[k], (what, k)


def differs(a, b):
    return a.keys() != b.keys() or any(not np.array_equal(a[k], b[k]) for k in a if isinstance(a[k], np.ndarray))


# ---------------------------------------------------------------- one edit, on a HostScene and in scene text

def apply_edit(scene, edit):
    """An edit (section, entity, keys) on a HostScene: Nodes -> set_node_shader (key shader), Shaders -> set_shader, Textures ->
    set_texture, Lights -> set_light, "place" -> place_node (a node edit, c2rt_scene_set_nodes)."""
    section, entity, keys = edit
    if section == "Nodes":
        scene.set_node_shader(entity, keys["shader"])
    elif section == "Shaders":
        scene.set_shader(entity, **keys)
    elif section == "Textures":
        scene.set_texture(entity, **keys)
    elif section == "Lights":
        scene.set_light(entity, **keys)
    else:
        scene.place_node(entity, **keys)


def edit_text(text, edit):
    """The same edit written into scene text."""
    from sdl_edit import edit_node
    section, entity, keys = edit
    if section == "place":
        return edit_node(text, entity, **keys)
    keys = dict(keys)
    kind = keys.pop("kind", None)
    return edit_entity(text, section, entity, kind=kind, **keys)
