"""Partial frames after edits (c2rt_render_update) without a GPU: the frame cache's lifetime, argument checks that come before any
device is touched, the loud failure without a device, and the exported symbols.  The frames themselves are checked on the GPU
(tests/test_gpu_update.py)."""
import ctypes as C
import os

import numpy as np
import pytest

import chess2rt_b200 as c2
from chess2rt_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HAS_GPU = c2.device_count() > 0
NEW_SYMBOLS = ("c2rt_frame_cache_create", "c2rt_frame_cache_destroy", "c2rt_render_update")


def _frame_blocks():
    s = c2.HostScene(os.path.join(ROOT, "scenes", "lecture5.sdl"))
    s.set_frame_size(32, 16)
    return s.frame_blocks()


def test_frame_cache_create_and_destroy():
    caches = [c2.FrameCache() for _ in range(3)]
    assert all(k.handle for k in caches) and len({k.handle for k in caches}) == 3
    for k in caches:
        k.close()
        k.close()   # twice: a no-op
        assert k.handle is None
    api.lib.c2rt_frame_cache_destroy(None)   # NULL is a no-op
    assert api.lib.c2rt_frame_cache_create(None) == -1
    assert b"out is null" in api.lib.c2rt_last_error()


def test_null_scene_cache_or_planes_are_refused_before_any_device():
    cam, st = _frame_blocks()
    rgb = np.zeros((16, 32, 3), np.float32)
    argb = np.zeros((16, 32), np.uint32)
    k = c2.FrameCache()
    fake_scene = C.c_void_p(1)   # never dereferenced: the checks above the scene's use refuse first
    cases = [
        (None, k.handle, rgb, argb, "scene, camera and settings must be non-null"),
        (fake_scene, k.handle, None, None, "rgb and argb are both null"),
    ]
    for scene, cache, r, a, msg in cases:
        rc = api.lib.c2rt_render_update(scene, C.byref(cam), C.byref(st), cache, r.ctypes.data if r is not None else None,
                                        a.ctypes.data if a is not None else None, None, None)
        assert rc == -1 and msg.encode() in api.lib.c2rt_last_error(), (rc, api.lib.c2rt_last_error())
    with pytest.raises(c2.C2rtError, match="scene, camera and settings must be non-null"):
        c2.render_update(None, cam, st, None, rgb, argb)
    # the null cache on a stand-in scene handle: refused before the scene is used
    rc = api.lib.c2rt_render_update(fake_scene, C.byref(cam), C.byref(st), None, rgb.ctypes.data, None, None, None)
    assert rc == -1 and b"cache is null" in api.lib.c2rt_last_error()


@pytest.mark.skipif(HAS_GPU, reason="checks the failure without a device")
def test_without_a_gpu_the_call_fails_loudly():
    s = c2.HostScene(os.path.join(ROOT, "scenes", "lecture5.sdl"))
    s.set_frame_size(32, 16)
    cam, st = s.frame_blocks()
    rgb = np.zeros((16, 32, 3), np.float32)
    with pytest.raises(c2.C2rtError) as e:
        s.render_update()
    assert e.value.status == -3   # C2RT_ERR_CUDA: no CPU fallback
    k = c2.FrameCache()
    with pytest.raises(c2.C2rtError) as e:
        c2.render_update(C.c_void_p(1), cam, st, k, rgb)
    assert e.value.status == -3


def test_library_exports_the_update_symbols():
    for name in NEW_SYMBOLS:
        assert name in api.C_ABI_SYMBOLS
        assert hasattr(api.lib, name)
    assert hasattr(api.host_lib, "c2rt_host_render_update")
    f = api.lib.c2rt_render_update
    assert len(f.argtypes) == 8
    assert C.sizeof(api.UpdateInfo) == 16
