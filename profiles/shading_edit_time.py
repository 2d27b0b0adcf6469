"""Highlighting a piece and moving the light: host wall time from the start of an edit to a synchronised next frame, shading /
light edits in place (HostScene.set_node_shader / set_light: c2rt_scene_set_node_shaders / c2rt_scene_set_lights) against
destroying the scene and creating it again from the edited description (what a host had to do before).  Every variant ends in
the same blocking ARGB-only frame (c2rt_render, rgb NULL: the interactive loop's delivery) and every repetition switches
between two states, so each edit changes the scene.  The variants alternate within each repetition; medians over --steps
repetitions.  Prints the device name, power limit and max SM clock with the numbers.

  python profiles/shading_edit_time.py [--steps 25] [--warmup 3] [--out result.json]

Workloads (1920x1080):
  chessboard_highlight  pawn e2 pointed at a spare "highlight" shader and back (a shader added to the scene text)
  lecture5_relight      the light moved between two positions
Variants:
  edit        the edit in place, then the frame
  create      the same edit in the flat description, c2rt_scene_destroy + c2rt_scene_create from it, then the frame
  frame_only  the frame alone
"""
import argparse
import ctypes as C
import json
import os
import shutil
import statistics
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from edit_time import device_info  # noqa: E402

HIGHLIGHT = '    Phong "highlight" {\n      color 0.25 0.875 0.25\n      exponent 20\n    }\n'


def chessboard_with_highlight(tmp):
    with open(os.path.join(ROOT, "scenes", "chessboard.sdl")) as fh:
        text = fh.read()
    i = text.index("Shaders {") + len("Shaders {\n")
    path = os.path.join(tmp, "chessboard_highlight.sdl")
    with open(path, "w") as fh:
        fh.write(text[:i] + HIGHLIGHT + text[i:])
    return path


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=25)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import chess2rt_b200 as c2
    from chess2rt_b200 import api

    if c2.device_count() < 1:
        raise SystemExit("shading_edit_time.py needs a CUDA device: libc2rt.so has no CPU fallback")
    c2.init(1, [0])
    name, limits = device_info()
    results = {"device": name, "power_limit_and_max_sm_clock": limits, "steps": args.steps, "warmup": args.warmup,
               "unit": "ms host wall time, edit start to synchronised ARGB frame, median", "workloads": {}}
    tmp = tempfile.mkdtemp(prefix="c2rt_shading_edit_")
    workloads = {
        # name: (scene file, the edit between two states on a HostScene)
        "chessboard_highlight_1080p": (chessboard_with_highlight(tmp),
                                       lambda s, r: s.set_node_shader("e2", ("white_piece", "highlight")[r % 2])),
        "lecture5_relight_1080p": (os.path.join(ROOT, "scenes", "lecture5.sdl"),
                                   lambda s, r: s.set_light("light1", pos=((-90.0, 700.0, 350.0), (150.0, 500.0, 200.0))[r % 2])),
    }
    w, h = 1920, 1080
    for wl, (path, edit) in workloads.items():
        # a: the scene edited in place; b: its flat description, re-created from after every edit
        a, b = c2.HostScene(path), c2.HostScene(path)
        for s in (a, b):
            s.set_frame_size(w, h)
        cam, st = a.frame_blocks()
        argb = np.empty((h, w), np.uint32)
        api.lib.c2rt_pin_host_buffer(argb.ctypes.data, argb.nbytes)
        ha = a.device_scene()
        hb = C.c_void_p()
        assert api.lib.c2rt_scene_create(b.desc(), C.byref(hb)) == 0, api.lib.c2rt_last_error()

        def frame(handle):
            rc = api.lib.c2rt_render(handle, C.byref(cam), C.byref(st), None, argb.ctypes.data, None)
            assert rc == 0, api.lib.c2rt_last_error()

        def edit_variant(r):
            edit(a, r)
            frame(ha)

        def create_variant(r):
            edit(b, r)
            api.lib.c2rt_scene_destroy(hb)
            assert api.lib.c2rt_scene_create(b.desc(), C.byref(hb)) == 0, api.lib.c2rt_last_error()
            frame(hb)

        def frame_variant(r):
            frame(ha)

        variants = {"edit": edit_variant, "create": create_variant, "frame_only": frame_variant}
        times = {k: [] for k in variants}
        for r in range(args.warmup + args.steps):
            for k, fn in variants.items():
                t0 = time.perf_counter()
                fn(r + 1)
                dt = (time.perf_counter() - t0) * 1e3
                if r >= args.warmup:
                    times[k].append(dt)
        res = {k: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v)} for k, v in times.items()}
        results["workloads"][wl] = res
        print(json.dumps({"workload": wl, "device": name, "limits": limits, **{k: round(v["median_ms"], 4) for k, v in res.items()}}),
              flush=True)
        api.lib.c2rt_scene_destroy(hb)
        api.lib.c2rt_unpin_host_buffer(argb.ctypes.data)
        a.close()
        b.close()
    c2.shutdown()
    shutil.rmtree(tmp)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(results, fh, indent=1)


if __name__ == "__main__":
    main()
