"""Multi-device path of c2rt_render (c2rt_init(N)): every device copies its interleaved bands to the host
frame itself, and the frame must be the same, bit for bit, as one device's — float frame, ARGB plane
(also delivered alone) and ray counts.  "distinct" needs >= 2 GPUs.  The other cases list device 0 two or
three times: each listing is a context of its own (streams, buffers, helper thread, bands), so the
multi-device code runs on a one-GPU box too."""
import os

import numpy as np
import pytest

import chess2rt_b200 as c2

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SC = os.path.join(ROOT, "scenes")


def _render(scene, size):
    h = c2.HostScene(os.path.join(SC, scene))
    h.set_frame_size(*size)
    rgb, argb, st = h.render(argb=True, count_rays=True)
    _, argb_only, st_a = h.render(argb_only=True, count_rays=True)
    h.close()
    return rgb, argb, st, argb_only, st_a


@pytest.mark.parametrize("devices", ["distinct", "dev0x2", "dev0x3"])
@pytest.mark.parametrize("scene,size", [("lecture5.sdl", (333, 217)), ("chessboard.sdl", (640, 360)), ("lecture4.sdl", (64, 1100))])
def test_single_process_multi_device_frame_is_bit_identical(scene, size, devices):
    if devices == "distinct":
        n = c2.device_count()
        if n < 2:
            pytest.skip("needs >= 2 GPUs")
        configs = [(k, None) for k in sorted({2, min(n, 4), n})]
    else:
        k = int(devices[-1])
        configs = [(k, [0] * k)]
    try:
        c2.init(1, [0])
        ref, ref_a, st1, ref_ao, st1_a = _render(scene, size)
        for k, ids in configs:
            c2.init(k, ids)
            rgb, argb, st, argb_only, st_a = _render(scene, size)
            for s in (st, st_a):
                assert s.n_gpus == k and s.launches >= k
            np.testing.assert_array_equal(rgb, ref)
            np.testing.assert_array_equal(argb, ref_a)
            np.testing.assert_array_equal(argb_only, ref_ao)
            assert (st.primary_rays, st.shadow_rays) == (st1.primary_rays, st1.shadow_rays)
            assert (st_a.primary_rays, st_a.shadow_rays) == (st1_a.primary_rays, st1_a.shadow_rays)
    finally:
        c2.init(1, [0])
