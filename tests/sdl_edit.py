"""Node edits written into scene text: the scene file a host would have loaded after moving, capturing or promoting a piece.
The edit tests compare HostScene.place_node / c2rt_scene_set_nodes against a scene loaded fresh from that text."""
import os
import re

import numpy as np

import chess2rt_b200 as c2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SC = os.path.join(ROOT, "scenes")
TSC = os.path.join(ROOT, "tests", "scenes")

_TRANSFORM_KEYS = ("scale", "rotate", "translate")


def _node_blocks(text):
    """(start of the body, end of the body, node name) of every `Node [name] { ... }` block."""
    out = []
    for m in re.finditer(r'\bNode\b\s*("([^"]*)")?\s*\{', text):
        depth, i = 1, m.end()
        while depth:
            depth += {"{": 1, "}": -1}.get(text[i], 0)
            i += 1
        body = text[m.end():i - 1]
        name = m.group(2)
        if name is None:
            nm = re.search(r'\bname\s+"([^"]*)"', body)
            name = nm.group(1) if nm else None
        out.append((m.end(), i - 1, name))
    return out


def edit_node(text, node, geometry=None, scale=None, rotate=None, translate=None):
    """`text` with node `node`'s entry edited as HostScene.place_node edits the loaded scene: `geometry` replaces the geometry
    key (None keeps it), and the scale / rotate / translate keys are replaced by the given ones (None: the key is dropped)."""
    for start, end, name in _node_blocks(text):
        if name != node:
            continue
        stmts = [s.strip() for s in re.split(r"[;\n]", text[start:end])]
        keep = [s for s in stmts if s and not s.startswith("//") and s.split()[0] not in _TRANSFORM_KEYS
                and not (geometry is not None and s.split()[0] == "geometry")]
        if geometry is not None:
            keep.append('geometry "%s"' % geometry)
        for key, v in zip(_TRANSFORM_KEYS, (scale, rotate, translate)):
            if v is not None:
                keep.append("%s %s" % (key, " ".join(repr(float(x)) for x in v)))
        return text[:start] + "\n      " + "\n      ".join(keep) + "\n    " + text[end:]
    raise KeyError(node)


def write_scene(tmp_dir, src_path, text):
    """Writes `text` as a scene file next to links to everything in the source scene's directory (bitmaps, skyboxes), so the
    relative paths in the text resolve as they do for the source file."""
    src_dir = os.path.dirname(os.path.abspath(src_path))
    for f in os.listdir(src_dir):
        dst = os.path.join(tmp_dir, f)
        if not os.path.lexists(dst):
            os.symlink(os.path.join(src_dir, f), dst)
    path = os.path.join(tmp_dir, "edited_" + os.path.basename(src_path))
    with open(path, "w") as fh:
        fh.write(text)
    return path


def load_edited(tmp_dir, src_path, edits):
    """A HostScene of `src_path` with each (node, kwargs) of `edits` written into its text."""
    with open(src_path) as fh:
        text = fh.read()
    for node, kw in edits:
        text = edit_node(text, node, **kw)
    return c2.HostScene(write_scene(tmp_dir, src_path, text))


# the arrays of a c2rt_scene_desc: (count field, array field, elements per entry, element type)
DESC_ARRAYS = [
    ("n_nodes", "node_geom", 1), ("n_nodes", "node_shader", 1), ("n_nodes", "node_transform", 9), ("n_nodes", "node_inverse", 9),
    ("n_nodes", "node_inverse_t", 9), ("n_nodes", "node_offset", 3),
    ("n_geoms", "geom_type", 1), ("n_geoms", "geom_params", 4), ("n_geoms", "geom_left", 1), ("n_geoms", "geom_right", 1),
    ("n_shaders", "shader_type", 1), ("n_shaders", "shader_color", 3), ("n_shaders", "shader_texture", 1),
    ("n_shaders", "shader_exponent", 1), ("n_shaders", "shader_strength", 1),
    ("n_textures", "tex_type", 1), ("n_textures", "tex_colors", 18), ("n_textures", "tex_params", 6), ("n_textures", "tex_width", 1),
    ("n_textures", "tex_height", 1), ("n_textures", "tex_texel_offset", 1), ("n_texels", "texels", 3),
    ("n_lights", "light_pos", 3), ("n_lights", "light_color", 3), ("n_lights", "light_power", 1),
]


def desc_arrays(scene):
    """Every array of the scene's flat description (copies), keyed by field name, plus the environment block."""
    d = scene.desc().contents
    out = {}
    for count, field, per in DESC_ARRAYS:
        n = getattr(d, count) * per
        p = getattr(d, field)
        out[field] = np.ctypeslib.as_array(p, (n,)).copy() if n else np.zeros(0)
    out["env"] = np.array([d.env_type] + list(d.env_face_width) + list(d.env_face_height) + list(d.env_face_texel_offset))
    return out


def assert_same_desc(a, b):
    """Array for array, bit for bit (NaN payloads included)."""
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape, k
        assert a[k].tobytes() == b[k].tobytes(), k
