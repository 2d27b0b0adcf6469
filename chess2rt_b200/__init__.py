"""chess2rt_b200 — B200-native (sm_100a) implementation of Chess2RT's per-pixel render loop.

The product is ``libc2rt.so`` (hand-written CUDA kernels behind the C ABI of ``include/c2rt.h``)
plus ``libc2rt_host.so`` (C++ mirror of the reference's scene API: loaders, object model, scene
flattener, renderer entry points).  This Python package is a thin ctypes harness over those two
libraries for tests and ``bench.py``; it contains no rendering code and no CPU fallback — touching
any attribute of :mod:`chess2rt_b200.api` raises if the libraries have not been built
(``python -m chess2rt_b200.build``).
"""
_API_NAMES = (
    "C2rtError", "HostScene", "HitPlanes", "Stats", "band_rows_owned", "device_count", "init", "lib", "host_lib", "render_device",
    "render_hits_device", "RayHits", "trace_rays_device", "test_visibility_device", "shade_rays_device", "scene_set_nodes", "scene_set_node_shaders", "scene_set_shaders",
    "scene_set_textures", "scene_set_lights", "read_ray_counters", "deinterleave", "measure_fma_peak", "srgb_table", "rng_u31", "shutdown",
    "FrameCache", "render_update",
)


def __getattr__(name):  # lazy: `python -m chess2rt_b200.build` must work before the libraries exist
    if name in _API_NAMES:
        from . import api
        return getattr(api, name)
    raise AttributeError(name)
