"""ctypes bindings of include/c2rt.h (libc2rt.so) and of the host mirror (libc2rt_host.so)."""
import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))


class C2rtError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"c2rt status {status}: {message}")
        self.status = status


def _load(name):
    path = os.path.join(os.environ.get("C2RT_LIB_DIR") or _PKG, name)  # C2RT_LIB_DIR: tuning variants (build.build_variant)
    if not os.path.exists(path):
        raise ImportError(
            f"{path} is missing: build it with `python -m chess2rt_b200.build` (or __graft_entry__.build()). "
            "There is no Python/CPU fallback for the render path.")
    return C.CDLL(path, mode=C.RTLD_GLOBAL)


lib = _load("libc2rt.so")
host_lib = _load("libc2rt_host.so")


class Camera(C.Structure):
    _fields_ = [("pos", C.c_double * 3), ("up_left", C.c_double * 3), ("up_right", C.c_double * 3),
                ("down_left", C.c_double * 3), ("right_dir", C.c_double * 3), ("up_dir", C.c_double * 3),
                ("front_dir", C.c_double * 3), ("frame_width", C.c_uint32), ("frame_height", C.c_uint32),
                ("dof", C.c_int32), ("num_samples", C.c_uint32), ("focal_plane_dist", C.c_double),
                ("disc_multiplier", C.c_double), ("stereo_separation", C.c_double)]


class Settings(C.Structure):
    _fields_ = [("frame_width", C.c_uint32), ("frame_height", C.c_uint32), ("aa_enabled", C.c_int32),
                ("gi_enabled", C.c_int32), ("prepass_enabled", C.c_int32), ("prepass_only", C.c_int32),
                ("max_trace_depth", C.c_uint32), ("ambient_light", C.c_float * 3), ("rng_seed", C.c_uint64),
                ("count_rays", C.c_int32), ("bucket_size", C.c_uint32),
                ("paths_per_pixel", C.c_uint32), ("reserved", C.c_uint32)]


class Band(C.Structure):
    _fields_ = [("rank", C.c_uint32), ("n_ranks", C.c_uint32), ("band_rows", C.c_uint32), ("compact", C.c_uint32),
                ("done_flags", C.c_void_p), ("frame_no", C.c_uint32), ("reserved", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [("kernel_ms", C.c_double), ("total_ms", C.c_double), ("primary_rays", C.c_uint64),
                ("shadow_rays", C.c_uint64), ("n_gpus", C.c_uint32), ("launches", C.c_uint32)]


class UpdateInfo(C.Structure):
    """c2rt_update_info: the tiles of a c2rt_render_update"""
    _fields_ = [("tiles_total", C.c_uint32), ("tiles_rendered", C.c_uint32), ("full", C.c_uint32), ("reserved", C.c_uint32)]

    def as_dict(self):
        return {"tiles_total": self.tiles_total, "tiles_rendered": self.tiles_rendered, "full": bool(self.full)}


class Hit(C.Structure):
    _fields_ = [("node", C.c_int32), ("reserved", C.c_int32), ("dist", C.c_double), ("p", C.c_double * 3),
                ("normal", C.c_double * 3), ("u", C.c_double), ("v", C.c_double)]


class HitPlanes(C.Structure):
    _fields_ = [("node", C.c_void_p), ("dist", C.c_void_p), ("normal", C.c_void_p), ("uv", C.c_void_p)]


class RayHits(C.Structure):
    _fields_ = [("node", C.c_void_p), ("dist", C.c_void_p), ("p", C.c_void_p), ("normal", C.c_void_p), ("uv", C.c_void_p)]


class SceneDesc(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("abi_version", C.c_uint32),
        ("n_nodes", C.c_uint32), ("node_geom", C.POINTER(C.c_int32)), ("node_shader", C.POINTER(C.c_int32)),
        ("node_transform", C.POINTER(C.c_double)), ("node_inverse", C.POINTER(C.c_double)),
        ("node_inverse_t", C.POINTER(C.c_double)), ("node_offset", C.POINTER(C.c_double)),
        ("n_geoms", C.c_uint32), ("geom_type", C.POINTER(C.c_int32)), ("geom_params", C.POINTER(C.c_double)),
        ("geom_left", C.POINTER(C.c_int32)), ("geom_right", C.POINTER(C.c_int32)),
        ("n_shaders", C.c_uint32), ("shader_type", C.POINTER(C.c_int32)), ("shader_color", C.POINTER(C.c_float)),
        ("shader_texture", C.POINTER(C.c_int32)), ("shader_exponent", C.POINTER(C.c_double)),
        ("shader_strength", C.POINTER(C.c_float)),
        ("n_textures", C.c_uint32), ("tex_type", C.POINTER(C.c_int32)), ("tex_colors", C.POINTER(C.c_float)),
        ("tex_params", C.POINTER(C.c_double)), ("tex_width", C.POINTER(C.c_int32)), ("tex_height", C.POINTER(C.c_int32)),
        ("tex_texel_offset", C.POINTER(C.c_uint64)), ("texels", C.POINTER(C.c_float)), ("n_texels", C.c_uint64),
        ("n_lights", C.c_uint32), ("light_pos", C.POINTER(C.c_double)), ("light_color", C.POINTER(C.c_float)),
        ("light_power", C.POINTER(C.c_float)),
        ("env_type", C.c_int32), ("env_reserved", C.c_int32), ("env_face_width", C.c_int32 * 6), ("env_face_height", C.c_int32 * 6),
        ("env_face_texel_offset", C.c_uint64 * 6),
    ]


# every symbol include/c2rt.h declares (tests/test_abi.py checks the library exports them all)
C_ABI_SYMBOLS = [
    "c2rt_init", "c2rt_shutdown", "c2rt_abi_version", "c2rt_device_count", "c2rt_last_error",
    "c2rt_scene_create", "c2rt_scene_destroy", "c2rt_scene_set_nodes", "c2rt_scene_set_node_shaders", "c2rt_scene_set_shaders",
    "c2rt_scene_set_textures", "c2rt_scene_set_lights", "c2rt_render", "c2rt_cancel", "c2rt_render_device", "c2rt_read_ray_counters",
    "c2rt_deinterleave", "c2rt_render_pixel", "c2rt_render_hits", "c2rt_render_hits_device",
    "c2rt_trace_rays", "c2rt_trace_rays_device", "c2rt_test_visibility", "c2rt_test_visibility_device",
    "c2rt_shade_rays", "c2rt_shade_rays_device", "c2rt_band_rows_owned", "c2rt_rng_u31", "c2rt_srgb_table",
    "c2rt_frame_alloc", "c2rt_frame_free", "c2rt_frame_export", "c2rt_frame_import", "c2rt_frame_unimport", "c2rt_frame_memset", "c2rt_frame_download", "c2rt_pin_host_buffer", "c2rt_unpin_host_buffer", "c2rt_gate",
    "c2rt_measure_fma_peak", "c2rt_selftest_device_pool", "c2rt_selftest_scene_class",
    "c2rt_frame_cache_create", "c2rt_frame_cache_destroy", "c2rt_render_update",
]

lib.c2rt_last_error.restype = C.c_char_p
lib.c2rt_selftest_device_pool.argtypes = [C.c_int, C.c_int]
lib.c2rt_selftest_device_pool.restype = C.c_longlong
lib.c2rt_init.argtypes = [C.c_int, C.POINTER(C.c_int)]
lib.c2rt_scene_create.argtypes = [C.POINTER(SceneDesc), C.POINTER(C.c_void_p)]
lib.c2rt_scene_destroy.argtypes = [C.c_void_p]
lib.c2rt_scene_destroy.restype = None
lib.c2rt_scene_set_nodes.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p]
lib.c2rt_scene_set_node_shaders.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
lib.c2rt_scene_set_shaders.argtypes = [C.c_void_p, C.c_size_t] + [C.c_void_p] * 6
lib.c2rt_scene_set_textures.argtypes = [C.c_void_p, C.c_size_t] + [C.c_void_p] * 3
lib.c2rt_scene_set_lights.argtypes = [C.c_void_p, C.c_size_t] + [C.c_void_p] * 4
lib.c2rt_render.argtypes = [C.c_void_p, C.POINTER(Camera), C.POINTER(Settings), C.c_void_p, C.c_void_p, C.POINTER(Stats)]
lib.c2rt_frame_cache_create.argtypes = [C.POINTER(C.c_void_p)]
lib.c2rt_frame_cache_destroy.argtypes = [C.c_void_p]
lib.c2rt_frame_cache_destroy.restype = None
lib.c2rt_render_update.argtypes = [C.c_void_p, C.POINTER(Camera), C.POINTER(Settings), C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.POINTER(Stats), C.POINTER(UpdateInfo)]
lib.c2rt_render_device.argtypes = [C.c_void_p, C.POINTER(Camera), C.POINTER(Settings), C.POINTER(Band), C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.POINTER(Stats)]
lib.c2rt_read_ray_counters.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
lib.c2rt_deinterleave.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                  C.c_uint32, C.c_void_p]
lib.c2rt_render_pixel.argtypes = [C.c_void_p, C.POINTER(Camera), C.POINTER(Settings), C.c_int, C.c_int,
                                  C.POINTER(C.c_float), C.POINTER(Hit)]
lib.c2rt_render_hits.argtypes = [C.c_void_p, C.POINTER(Camera), C.POINTER(Settings), C.POINTER(HitPlanes), C.POINTER(Stats)]
lib.c2rt_render_hits_device.argtypes = [C.c_void_p, C.POINTER(Camera), C.POINTER(Settings), C.POINTER(Band), C.POINTER(HitPlanes),
                                        C.c_void_p, C.POINTER(Stats)]
lib.c2rt_trace_rays.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.POINTER(RayHits), C.POINTER(Stats)]
lib.c2rt_trace_rays_device.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.POINTER(RayHits), C.c_void_p,
                                       C.POINTER(Stats)]
lib.c2rt_test_visibility.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Stats)]
lib.c2rt_test_visibility_device.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.POINTER(Stats)]
lib.c2rt_shade_rays.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.POINTER(Stats)]
lib.c2rt_shade_rays_device.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.POINTER(Stats)]
lib.c2rt_band_rows_owned.argtypes = [C.c_uint32] * 4
lib.c2rt_band_rows_owned.restype = C.c_uint32
lib.c2rt_rng_u31.argtypes = [C.c_uint64] + [C.c_uint32] * 5
lib.c2rt_rng_u31.restype = C.c_uint32
lib.c2rt_srgb_table.argtypes = [C.c_void_p]
lib.c2rt_srgb_table.restype = None
lib.c2rt_frame_alloc.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
lib.c2rt_frame_free.argtypes = [C.c_void_p]
lib.c2rt_frame_export.argtypes = [C.c_void_p, C.c_void_p]
lib.c2rt_frame_import.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
lib.c2rt_frame_unimport.argtypes = [C.c_void_p]
lib.c2rt_frame_memset.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_void_p]
lib.c2rt_frame_download.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
lib.c2rt_pin_host_buffer.argtypes = [C.c_void_p, C.c_size_t]
lib.c2rt_unpin_host_buffer.argtypes = [C.c_void_p]
lib.c2rt_gate.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
lib.c2rt_measure_fma_peak.argtypes = [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]

host_lib.c2rt_host_last_error.restype = C.c_char_p
host_lib.c2rt_host_scene_load.argtypes = [C.c_char_p]
host_lib.c2rt_host_scene_load.restype = C.c_void_p
host_lib.c2rt_host_scene_free.argtypes = [C.c_void_p]
host_lib.c2rt_host_scene_free.restype = None
host_lib.c2rt_host_scene_set_frame_size.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
host_lib.c2rt_host_scene_set_frame_size.restype = None
host_lib.c2rt_host_scene_get_frame_size.argtypes = [C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
host_lib.c2rt_host_scene_get_frame_size.restype = None
host_lib.c2rt_host_scene_override.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
host_lib.c2rt_host_scene_override.restype = None
host_lib.c2rt_host_scene_desc.argtypes = [C.c_void_p]
host_lib.c2rt_host_scene_desc.restype = C.POINTER(SceneDesc)
host_lib.c2rt_host_scene_place_node.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p]
host_lib.c2rt_host_scene_index.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
host_lib.c2rt_host_scene_name.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
host_lib.c2rt_host_scene_name.restype = C.c_char_p
host_lib.c2rt_host_scene_set_node_shader.argtypes = [C.c_void_p, C.c_int, C.c_char_p]
host_lib.c2rt_host_scene_set_shader.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p]
host_lib.c2rt_host_scene_set_texture.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 8
host_lib.c2rt_host_scene_set_light.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
host_lib.c2rt_host_frame_blocks.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.POINTER(Camera), C.POINTER(Settings)]
host_lib.c2rt_host_frame_blocks.restype = None
host_lib.c2rt_host_device_scene.argtypes = [C.c_void_p]
host_lib.c2rt_host_device_scene.restype = C.c_void_p
host_lib.c2rt_host_render.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.POINTER(Stats)]
host_lib.c2rt_host_render_update.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.POINTER(Stats),
                                            C.POINTER(UpdateInfo)]
host_lib.c2rt_host_render_pixel.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(Hit)]
host_lib.c2rt_host_render_hits.argtypes = [C.c_void_p, C.POINTER(HitPlanes), C.c_uint64, C.POINTER(Stats)]
host_lib.c2rt_host_trace_rays.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.POINTER(RayHits), C.POINTER(Stats)]
host_lib.c2rt_host_test_visibility.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Stats)]
host_lib.c2rt_host_shade_rays.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Stats)]
host_lib.c2rt_host_camera_rotate.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double]
host_lib.c2rt_host_camera_rotate.restype = None
host_lib.c2rt_host_camera_move.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double]
host_lib.c2rt_host_camera_move.restype = None
host_lib.c2rt_host_save_bmp.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p, C.c_size_t]
host_lib.c2rt_host_save_bmp.restype = C.c_size_t
host_lib.c2rt_host_scene_info.argtypes = [C.c_void_p, C.POINTER(C.c_int32)]
host_lib.c2rt_host_scene_info.restype = None
host_lib.c2rt_host_decode_bmp.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.c_void_p,
                                          C.c_size_t]


def _check(rc):
    if rc != 0:
        raise C2rtError(rc, lib.c2rt_last_error().decode())


def _check_host(rc):
    if rc != 0:
        raise C2rtError(rc, host_lib.c2rt_host_last_error().decode())


def device_count():
    return lib.c2rt_device_count()


def init(n_gpus=1, device_ids=None):
    ids = (C.c_int * n_gpus)(*device_ids) if device_ids is not None else None
    _check(lib.c2rt_init(n_gpus, ids))


def shutdown():
    lib.c2rt_shutdown()


def band_rows_owned(height, rank, n_ranks, band_rows):
    return lib.c2rt_band_rows_owned(height, rank, n_ranks, band_rows)


def rng_u31(seed, px, py, tap, sample, draw):
    return lib.c2rt_rng_u31(seed, px, py, tap, sample, draw)


def srgb_table():
    out = np.zeros(4097, np.uint8)
    lib.c2rt_srgb_table(out.ctypes.data)
    return out


def measure_fma_peak(fp64=False):
    tf, mhz = C.c_double(), C.c_double()
    _check(lib.c2rt_measure_fma_peak(int(fp64), C.byref(tf), C.byref(mhz)))
    return tf.value, mhz.value


class HostScene:
    """A scene file loaded by the reference-compatible host loader (rt::parseSceneFromFile)."""

    def __init__(self, path):
        self._h = host_lib.c2rt_host_scene_load(os.fspath(path).encode())
        if not self._h:
            raise C2rtError(-1, host_lib.c2rt_host_last_error().decode())
        self.path = os.fspath(path)

    def close(self):
        if self._h:
            host_lib.c2rt_host_scene_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_frame_size(self, w, h):
        host_lib.c2rt_host_scene_set_frame_size(self._h, w, h)

    @property
    def frame_size(self):
        w, h = C.c_uint32(), C.c_uint32()
        host_lib.c2rt_host_scene_get_frame_size(self._h, C.byref(w), C.byref(h))
        return w.value, h.value

    def override(self, aa=-1, dof=-1, prepass=-1, num_samples=-1):
        host_lib.c2rt_host_scene_override(self._h, int(aa), int(dof), int(prepass), int(num_samples))

    def info(self):
        out = (C.c_int32 * 8)()
        host_lib.c2rt_host_scene_info(self._h, out)
        keys = ["nodes", "geometries", "shaders", "textures", "lights", "aa", "dof", "num_samples"]
        return dict(zip(keys, list(out)))

    def desc(self):
        p = host_lib.c2rt_host_scene_desc(self._h)
        if not p:
            raise C2rtError(-1, host_lib.c2rt_host_last_error().decode())
        return p

    def node_index(self, name):
        """The index of the node the scene file names `name` (its place in the description's node arrays)."""
        return self.index("nodes", str(name))

    def place_node(self, node, geometry=None, scale=None, rotate=None, translate=None):
        """As if the node's entry in the scene file had been edited: `geometry` (a geometry name; None keeps it) and the keys
        scale / rotate / translate (three numbers each; None: the key is absent).  The node's Transform is reset and the keys
        are applied as the loader applies them.  `node` is a node name or index.  The flat description and any uploaded scene
        follow (c2rt_scene_set_nodes), so the next frame shows the edit.  A bad node or geometry name changes nothing."""
        i = self.node_index(node) if isinstance(node, str) else int(node)
        for v, name in zip((scale, rotate, translate), ("scale", "rotate", "translate")):
            if v is not None and len(v) != 3:
                raise ValueError(f"{name} needs three numbers, got {len(v)}")
        vecs = [None if v is None else (C.c_double * 3)(*[float(x) for x in v]) for v in (scale, rotate, translate)]
        _check_host(host_lib.c2rt_host_scene_place_node(self._h, i, None if geometry is None else str(geometry).encode(), *vecs))

    def index(self, section, entity):
        """The index of an entity of `section` ("nodes", "shaders", "textures" or "lights"): its place in the description's
        arrays.  `entity` is the name the scene file gives it, or an index (checked by the edit that takes it)."""
        if not isinstance(entity, str):
            return int(entity)
        i = host_lib.c2rt_host_scene_index(self._h, section.encode(), entity.encode())
        if i < 0:
            raise KeyError(f"no {section[:-1]} named {entity!r}")
        return i

    def set_node_shader(self, node, shader):
        """As if the node's `shader` key in the scene file named `shader` (a shader name or index): highlighting a piece and
        back.  The flat description and any uploaded scene follow (c2rt_scene_set_node_shaders).  A bad name changes nothing."""
        i = self.index("nodes", node)
        _check_host(host_lib.c2rt_host_scene_set_node_shader(self._h, i, self._name("shaders", shader).encode()))

    def set_shader(self, shader, kind=None, color=None, texture=..., exponent=None, strength=None):
        """As if the shader's entry in the scene file had been edited.  kind ("Lambert" or "Phong"; None keeps the object)
        replaces it with a fresh shader of that kind, with that kind's defaults; then the given keys apply as the loader applies
        them: color (three numbers), texture (a texture name or index; None for no texture; omitted: kept), exponent and
        strength (Phong keys, clamped as the loader clamps them).  `shader` is a name or index.  The flat description and any
        uploaded scene follow (c2rt_scene_set_shaders).  A bad name, index, kind or key changes nothing."""
        i = self.index("shaders", shader)
        tex = None if texture is ... else ("" if texture is None else self._name("textures", texture))
        _check_host(host_lib.c2rt_host_scene_set_shader(
            self._h, i, None if kind is None else str(kind).encode(), _floats(color, 3, "color"),
            None if tex is None else tex.encode(), _doubles(exponent, 1, "exponent"), _floats(strength, 1, "strength")))

    def set_texture(self, texture, color1=None, color2=None, size=None, colorU=None, colorV=None, freqU=None, freqV=None,
                    scaling=None):
        """As if the texture's entry in the scene file had the given keys replaced (None: kept).  Checker: color1, color2 (three
        numbers each), size; Procedure2: colorU, colorV (three colours), freqU, freqV (three numbers each); BitmapTexture:
        scaling.  A texture keeps its kind and its bitmap.  `texture` is a name or index.  The flat description and any uploaded
        scene follow (c2rt_scene_set_textures).  A bad name or index, or a key of another kind, changes nothing."""
        i = self.index("textures", texture)
        _check_host(host_lib.c2rt_host_scene_set_texture(
            self._h, i, _floats(color1, 3, "color1"), _floats(color2, 3, "color2"), _doubles(size, 1, "size"),
            _floats(colorU, 9, "colorU"), _floats(colorV, 9, "colorV"), _doubles(freqU, 3, "freqU"), _doubles(freqV, 3, "freqV"),
            _floats(scaling, 1, "scaling")))

    def set_light(self, light, pos=None, color=None, power=None):
        """As if the light's entry in the scene file had the given keys replaced (None: kept): pos, color (three numbers each),
        power.  `light` is a name or index.  The flat description and any uploaded scene follow (c2rt_scene_set_lights).  A bad
        name or index changes nothing."""
        i = self.index("lights", light)
        _check_host(host_lib.c2rt_host_scene_set_light(self._h, i, _doubles(pos, 3, "pos"), _floats(color, 3, "color"),
                                                       _floats(power, 1, "power")))

    def _name(self, section, entity):
        """The scene file's name of an entity given by name or index (the host mirror's edits take references by name)."""
        if isinstance(entity, str):
            return entity
        p = host_lib.c2rt_host_scene_name(self._h, section.encode(), int(entity))
        if p is None:
            raise KeyError(f"{section[:-1]} {entity} does not exist or has no name")
        return p.decode()

    def frame_blocks(self, seed=0, count_rays=False):
        cam, st = Camera(), Settings()
        host_lib.c2rt_host_frame_blocks(self._h, seed, int(count_rays), C.byref(cam), C.byref(st))
        return cam, st

    def device_scene(self):
        p = host_lib.c2rt_host_device_scene(self._h)
        if not p:
            raise C2rtError(-3, host_lib.c2rt_host_last_error().decode())
        return p

    def render(self, argb=False, seed=0, count_rays=False, out=None, out_argb=None, argb_only=False):
        """Renderer(scene, output).renderRT() with HOST buffers -> (rgb[H,W,3] float32, argb[H,W] uint32|None, Stats).
        argb_only: no float frame is written or copied (rgb is None in the result)."""
        w, h = self.frame_size
        rgb = None if argb_only else (out if out is not None else np.empty((h, w, 3), np.float32))
        a = out_argb if out_argb is not None else (np.empty((h, w), np.uint32) if (argb or argb_only) else None)
        st = Stats()
        rc = host_lib.c2rt_host_render(self._h, rgb.ctypes.data if rgb is not None else None, a.ctypes.data if a is not None else None,
                                       seed, int(count_rays), C.byref(st))
        self.cancelled = rc == 1   # C2RT_CANCELLED: a c2rt_cancel reached the frame (partial image), not an error
        if rc != 1:
            _check_host(rc)
        return rgb, a, st

    def render_update(self, argb=False, argb_only=False, seed=0, count_rays=False):
        """render()'s frame, bit for bit, through the scene's frame cache (c2rt_render_update): after edits only the tiles they
        can have changed are rendered.  The frame goes into arrays this object keeps for the frame size and planes (the cache
        needs the buffers of the previous frame), so the returned arrays are overwritten by the next render_update: copy them
        to keep them.  -> (rgb[H,W,3] float32 | None with argb_only, argb[H,W] uint32 | None, Stats, info dict: tiles_total,
        tiles_rendered, full)"""
        w, h = self.frame_size
        key = (w, h, bool(argb or argb_only), bool(argb_only))
        if getattr(self, "_update_key", None) != key:   # new buffers: the next frame is a full one
            self._update_key = key
            self._update_rgb = None if argb_only else np.zeros((h, w, 3), np.float32)
            self._update_argb = np.zeros((h, w), np.uint32) if key[2] else None
        rgb, a = self._update_rgb, self._update_argb
        st, info = Stats(), UpdateInfo()
        rc = host_lib.c2rt_host_render_update(self._h, rgb.ctypes.data if rgb is not None else None,
                                              a.ctypes.data if a is not None else None, seed, int(count_rays), C.byref(st),
                                              C.byref(info))
        self.cancelled = rc == 1   # C2RT_CANCELLED (the cache starts over at the next call)
        if rc != 1:
            _check_host(rc)
        return rgb, a, st, info.as_dict()

    def camera_rotate(self, d_yaw, d_roll=0.0, d_pitch=0.0):
        host_lib.c2rt_host_camera_rotate(self._h, d_yaw, d_roll, d_pitch)

    def camera_move(self, dx, dy, dz):
        host_lib.c2rt_host_camera_move(self._h, dx, dy, dz)

    def render_pixel(self, x, y):
        rgb = (C.c_float * 3)()
        hit = Hit()
        _check_host(host_lib.c2rt_host_render_pixel(self._h, x, y, rgb, C.byref(hit)))
        return np.array(list(rgb), np.float32), hit


    def render_hits(self, planes=("node", "dist", "normal", "uv"), seed=0):
        """renderPixel's hit record for every pixel (c2rt_render_hits) -> ({plane: array}, Stats).  Planes: node [H, W] int32
        (-1 = miss), dist [H, W] float32 (+inf for a miss), normal [H, W, 3] and uv [H, W, 2] float32 (0 for a miss)."""
        w, h = self.frame_size
        out = {name: np.empty((h, w) + shape, dtype) for name, (dtype, shape) in HIT_PLANES.items() if name in planes}
        unknown = set(planes) - set(HIT_PLANES)
        if unknown:
            raise ValueError(f"unknown hit planes {sorted(unknown)}")
        p = HitPlanes(*(out[name].ctypes.data if name in out else None for name in HIT_PLANES))
        st = Stats()
        _check_host(host_lib.c2rt_host_render_hits(self._h, C.byref(p), seed, C.byref(st)))
        return out, st

    def trace_rays(self, origins, dirs, planes=("node", "dist", "p", "normal", "uv")):
        """The closest hit of every ray (origins[i], normalize(dirs[i])) (c2rt_trace_rays) -> ({plane: array}, Stats).  origins
        and dirs: [n, 3] float64.  Planes: node [n] int32 (-1 = miss), dist [n] (+inf for a miss), p, normal [n, 3] and uv
        [n, 2] float64 (0 for a miss)."""
        o, d = _points(origins), _points(dirs)
        if o.shape != d.shape:
            raise ValueError(f"origins {o.shape} and dirs {d.shape} differ in shape")
        unknown = set(planes) - set(RAY_PLANES)
        if unknown:
            raise ValueError(f"unknown ray planes {sorted(unknown)}")
        n = len(o)
        out = {name: np.empty((n,) + shape, dtype) for name, (dtype, shape) in RAY_PLANES.items() if name in planes}
        p = RayHits(*(out[name].ctypes.data if name in out else None for name in RAY_PLANES))
        st = Stats()
        _check_host(host_lib.c2rt_host_trace_rays(self._h, n, o.ctypes.data, d.ctypes.data, C.byref(p), C.byref(st)))
        return out, st

    def test_visibility(self, frm, to):
        """testVisibility(frm[i], to[i]) for every i (c2rt_test_visibility) -> (bool [n] array, Stats).  frm, to: [n, 3]."""
        f, t = _points(frm), _points(to)
        if f.shape != t.shape:
            raise ValueError(f"frm {f.shape} and to {t.shape} differ in shape")
        vis = np.empty(len(f), np.uint8)
        st = Stats()
        _check_host(host_lib.c2rt_host_test_visibility(self._h, len(f), f.ctypes.data, t.ctypes.data, vis.ctypes.data, C.byref(st)))
        return vis.astype(bool), st

    def shade_rays(self, origins, dirs, argb=False):
        """trace((origins[i], normalize(dirs[i]))) at depth 0 with the scene file's ambientLightColor (c2rt_shade_rays) ->
        (rgb [n, 3] float32, argb [n] uint32 (Color.toRGB32) or None, Stats).  origins and dirs: [n, 3] float64.  An untraced
        query (a non-finite coordinate, a zero direction) is (0, 0, 0) and 0."""
        o, d = _points(origins), _points(dirs)
        if o.shape != d.shape:
            raise ValueError(f"origins {o.shape} and dirs {d.shape} differ in shape")
        n = len(o)
        rgb = np.empty((n, 3), np.float32)
        a = np.empty(n, np.uint32) if argb else None
        st = Stats()
        _check_host(host_lib.c2rt_host_shade_rays(self._h, n, o.ctypes.data, d.ctypes.data, rgb.ctypes.data,
                                                  a.ctypes.data if a is not None else None, C.byref(st)))
        return rgb, a, st


def _floats(v, n, what):
    """None, or a C float array of the n numbers of v (a number when n == 1)."""
    return _array(v, n, what, C.c_float)


def _doubles(v, n, what):
    return _array(v, n, what, C.c_double)


def _array(v, n, what, ctype):
    if v is None:
        return None
    vals = np.asarray(v, np.float64).reshape(-1)
    if len(vals) != n:
        raise ValueError(f"{what} needs {n} numbers, got {len(vals)}")
    return C.cast((ctype * n)(*vals.tolist()), C.c_void_p)


def _points(a):
    a = np.ascontiguousarray(a, np.float64)
    if a.ndim != 2 or a.shape[1] != 3:
        raise ValueError(f"expected an [n, 3] array of points, got shape {a.shape}")
    return a


# the planes of a ray query: element type and per-ray shape, in c2rt_ray_hits order
RAY_PLANES = {"node": (np.int32, ()), "dist": (np.float64, ()), "p": (np.float64, (3,)), "normal": (np.float64, (3,)),
              "uv": (np.float64, (2,))}

# the planes of a hit frame: element type and per-pixel shape, in c2rt_hit_planes order
HIT_PLANES = {"node": (np.int32, ()), "dist": (np.float32, ()), "normal": (np.float32, (3,)), "uv": (np.float32, (2,))}


def save_bmp(argb, pad_rows=False):
    """saveBmp (imageio/bmp.d:195-237) of a packed uint32 plane [H, W] -> bytes."""
    a = np.ascontiguousarray(argb, np.uint32)
    h, w = a.shape
    out = np.zeros(54 + (w * 3 + 3) // 4 * 4 * h, np.uint8)
    n = host_lib.c2rt_host_save_bmp(a.ctypes.data, w, h, int(pad_rows), out.ctypes.data, out.size)
    return out[:n].tobytes()


def cancel():
    _check(lib.c2rt_cancel())


def scene_set_nodes(scene_handle, nodes, geom=None, transform=None, inverse=None, inverse_t=None, offset=None):
    """c2rt_scene_set_nodes on an uploaded scene (a handle from HostScene.device_scene or c2rt_scene_create): entry i sets node
    nodes[i]'s geometry index geom[i] and / or its transform[i], inverse[i], inverse_t[i] (3x3, row-major) and offset[i].  geom
    None keeps the geometries; the four transform arrays are given together or not at all."""
    ids = np.ascontiguousarray(nodes, np.uint32).reshape(-1)
    n = len(ids)
    g = None if geom is None else np.ascontiguousarray(geom, np.int32).reshape(-1)
    if g is not None and len(g) != n:
        raise ValueError(f"geom has {len(g)} entries for {n} nodes")
    tf = []
    for a, per in ((transform, 9), (inverse, 9), (inverse_t, 9), (offset, 3)):
        a = None if a is None else np.ascontiguousarray(a, np.float64).reshape(-1)
        if a is not None and len(a) != per * n:
            raise ValueError(f"a transform array has {len(a)} elements, {per * n} expected")
        tf.append(a)
    ptr = lambda a: None if a is None else a.ctypes.data  # noqa: E731
    _check(lib.c2rt_scene_set_nodes(scene_handle, n, ptr(ids), ptr(g), *[ptr(a) for a in tf]))


def _entries(a, n, per, dtype, what):
    a = np.ascontiguousarray(a, dtype).reshape(-1)
    if len(a) != per * n:
        raise ValueError(f"{what} has {len(a)} elements, {per * n} expected")
    return a


def scene_set_node_shaders(scene_handle, nodes, shader):
    """c2rt_scene_set_node_shaders on an uploaded scene: entry i points node nodes[i] at shader index shader[i] (description
    indices, as in c2rt_scene_desc)."""
    ids = np.ascontiguousarray(nodes, np.uint32).reshape(-1)
    sh = _entries(shader, len(ids), 1, np.int32, "shader")
    _check(lib.c2rt_scene_set_node_shaders(scene_handle, len(ids), ids.ctypes.data, sh.ctypes.data))


def scene_set_shaders(scene_handle, shaders, type, color, texture, exponent, strength):
    """c2rt_scene_set_shaders on an uploaded scene: entry i replaces shader shaders[i] with type[i] (C2RT_SHADER_*), color[i]
    (three floats), texture[i] (a texture index, < 0: none), exponent[i] and strength[i]."""
    ids = np.ascontiguousarray(shaders, np.uint32).reshape(-1)
    n = len(ids)
    arrs = [_entries(type, n, 1, np.int32, "type"), _entries(color, n, 3, np.float32, "color"),
            _entries(texture, n, 1, np.int32, "texture"), _entries(exponent, n, 1, np.float64, "exponent"),
            _entries(strength, n, 1, np.float32, "strength")]
    _check(lib.c2rt_scene_set_shaders(scene_handle, n, ids.ctypes.data, *[a.ctypes.data for a in arrs]))


def scene_set_textures(scene_handle, textures, colors, params):
    """c2rt_scene_set_textures on an uploaded scene: entry i replaces texture textures[i]'s colors[i] (18 floats) and params[i]
    (6 doubles), laid out as c2rt_scene_desc's tex_colors / tex_params; a bitmap reads params[i][0] (scaling) only."""
    ids = np.ascontiguousarray(textures, np.uint32).reshape(-1)
    n = len(ids)
    c, p = _entries(colors, n, 18, np.float32, "colors"), _entries(params, n, 6, np.float64, "params")
    _check(lib.c2rt_scene_set_textures(scene_handle, n, ids.ctypes.data, c.ctypes.data, p.ctypes.data))


def scene_set_lights(scene_handle, lights, pos, color, power):
    """c2rt_scene_set_lights on an uploaded scene: entry i replaces light lights[i]'s pos[i] (three doubles), color[i] (three
    floats, not premultiplied) and power[i]."""
    ids = np.ascontiguousarray(lights, np.uint32).reshape(-1)
    n = len(ids)
    arrs = [_entries(pos, n, 3, np.float64, "pos"), _entries(color, n, 3, np.float32, "color"), _entries(power, n, 1, np.float32, "power")]
    _check(lib.c2rt_scene_set_lights(scene_handle, n, ids.ctypes.data, *[a.ctypes.data for a in arrs]))


class FrameCache:
    """A c2rt_frame_cache for render_update (destroyed by close() or when collected)."""

    def __init__(self):
        h = C.c_void_p()
        _check(lib.c2rt_frame_cache_create(C.byref(h)))
        self.handle = h.value

    def close(self):
        if self.handle:
            lib.c2rt_frame_cache_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def render_update(scene_handle, cam, settings, cache, rgb, argb=None):
    """c2rt_render_update into HOST numpy arrays (rgb [H,W,3] float32 and argb [H,W] uint32, either None), which must hold what
    the previous render_update with `cache` (a FrameCache, or a raw handle) wrote into them -> (Stats, info dict).  A cancelled
    frame raises C2rtError with code 1."""
    st, info = Stats(), UpdateInfo()
    handle = cache.handle if isinstance(cache, FrameCache) else cache
    _check(lib.c2rt_render_update(scene_handle, C.byref(cam), C.byref(settings), handle, rgb.ctypes.data if rgb is not None else None,
                                  argb.ctypes.data if argb is not None else None, C.byref(st), C.byref(info)))
    return st, info.as_dict()


def render_device(scene_handle, cam, settings, d_rgb_ptr, d_argb_ptr=None, band=None, stream=None):
    """c2rt_render_device: device pointers (ints), async on `stream` (int cudaStream_t or None)."""
    b = C.byref(band) if band is not None else None
    _check(lib.c2rt_render_device(scene_handle, C.byref(cam), C.byref(settings), b, d_rgb_ptr, d_argb_ptr, stream, None))


def render_hits_device(scene_handle, cam, settings, node=None, dist=None, normal=None, uv=None, band=None, stream=None):
    """c2rt_render_hits_device: plane device pointers (ints, e.g. a torch tensor's data_ptr(); None = not wanted), async on
    `stream` (int cudaStream_t or None)."""
    b = C.byref(band) if band is not None else None
    p = HitPlanes(node, dist, normal, uv)
    _check(lib.c2rt_render_hits_device(scene_handle, C.byref(cam), C.byref(settings), b, C.byref(p), stream, None))


def trace_rays_device(scene_handle, n, d_origins, d_dirs, node=None, dist=None, p=None, normal=None, uv=None, stream=None):
    """c2rt_trace_rays_device: [n*3] float64 inputs and the output planes as device pointers (ints, e.g. a torch tensor's
    data_ptr(); None = not wanted), async on `stream` (int cudaStream_t or None)."""
    out = RayHits(node, dist, p, normal, uv)
    _check(lib.c2rt_trace_rays_device(scene_handle, n, d_origins, d_dirs, C.byref(out), stream, None))


def test_visibility_device(scene_handle, n, d_from, d_to, d_visible, stream=None):
    """c2rt_test_visibility_device: [n*3] float64 inputs and the [n] uint8 output as device pointers, async on `stream`."""
    _check(lib.c2rt_test_visibility_device(scene_handle, n, d_from, d_to, d_visible, stream, None))


def shade_rays_device(scene_handle, n, d_origins, d_dirs, ambient, d_rgb=None, d_argb=None, stream=None):
    """c2rt_shade_rays_device: [n*3] float64 inputs, the [n*3] float32 rgb and [n] uint32 argb outputs as device pointers (ints;
    None = not wanted), `ambient` three floats on the host, async on `stream` (int cudaStream_t or None)."""
    amb = (C.c_float * 3)(*ambient)
    _check(lib.c2rt_shade_rays_device(scene_handle, amb, n, d_origins, d_dirs, d_rgb, d_argb, stream, None))


def read_ray_counters(scene_handle, stream=None):
    p, s = C.c_uint64(), C.c_uint64()
    _check(lib.c2rt_read_ray_counters(scene_handle, stream, C.byref(p), C.byref(s)))
    return p.value, s.value


def deinterleave(gathered_ptr, frame_ptr, width, height, elem_words, n_ranks, band_rows, rows_pad, stream=None):
    _check(lib.c2rt_deinterleave(gathered_ptr, frame_ptr, width, height, elem_words, n_ranks, band_rows, rows_pad, stream))
