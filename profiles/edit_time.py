"""Moving pieces: host wall time from the start of an edit to a synchronised next frame, node edits in place
(c2rt_scene_set_nodes through HostScene.place_node, or one call for many nodes) against destroying the scene and creating it
again from the edited description (what a host had to do before).  Every variant ends in the same blocking ARGB-only frame
(c2rt_render, rgb NULL: the interactive loop's delivery) and every repetition moves the pieces between two positions, so
each edit changes the scene.  The variants alternate within each repetition; medians over --steps repetitions.  Prints the
device name, power limit and max SM clock with the numbers.

  python profiles/edit_time.py [--steps 25] [--warmup 3] [--out result.json]

Variants (chessboard, lecture5 at 1920x1080):
  edit_one      place_node of one node (pawn e2 / ball S1), then the frame
  create_one    the same node edit in the flat description, c2rt_scene_destroy + c2rt_scene_create from it, then the frame
  edit_all      (chessboard) the 32 pieces moved by one c2rt_scene_set_nodes call, then the frame
  create_all    (chessboard) the same 32 moves in the flat description, destroy + create, then the frame
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (scene file, width, height, node moved by the one-node variants, its two positions)
    "chessboard_1080p": ("scenes/chessboard.sdl", 1920, 1080, "e2", ((10.0, 0.0, -50.0), (10.0, 0.0, -10.0))),
    "lecture5_1080p": ("scenes/lecture5.sdl", 1920, 1080, "S1", ((100.0, 15.0, 256.0), (60.0, 15.0, 236.0))),
}


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


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
        raise SystemExit("edit_time.py needs a CUDA device: libc2rt.so has no CPU fallback")
    c2.init(1, [0])
    name, limits = device_info()
    results = {"device": name, "power_limit_and_max_sm_clock": limits, "steps": args.steps, "warmup": args.warmup,
               "unit": "ms host wall time, edit start to synchronised ARGB frame, median", "workloads": {}}
    for wl, (path, w, h, node, positions) in WORKLOADS.items():
        path = os.path.join(ROOT, path)
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

        def recreate():
            api.lib.c2rt_scene_destroy(hb)
            assert api.lib.c2rt_scene_create(b.desc(), C.byref(hb)) == 0, api.lib.c2rt_last_error()

        # the 32 pieces of the chessboard (every node but the floor), moved 5 units along z and back
        pieces = []
        if "chessboard" in wl:
            d = a.desc().contents
            pieces = list(range(1, d.n_nodes))
            off0 = np.array([[d.node_offset[3 * i + k] for k in range(3)] for i in pieces])
            mats = [np.array([[getattr(d, f)[9 * i + k] for k in range(9)] for i in pieces])
                    for f in ("node_transform", "node_inverse", "node_inverse_t")]
            geom = np.array([d.node_geom[i] for i in pieces], np.int32)
            offs = (off0, off0 + [0.0, 0.0, 5.0])

        def edit_one(r):
            a.place_node(node, translate=positions[r % 2])
            frame(ha)

        def create_one(r):
            b.place_node(node, translate=positions[r % 2])
            recreate()
            frame(hb)

        def edit_all(r):
            c2.scene_set_nodes(ha, pieces, geom=geom, transform=mats[0], inverse=mats[1], inverse_t=mats[2], offset=offs[r % 2])
            frame(ha)

        def create_all(r):
            dc = b.desc().contents
            for j, i in enumerate(pieces):
                for k in range(3):
                    dc.node_offset[3 * i + k] = float(offs[r % 2][j, k])
            recreate()
            frame(hb)

        variants = {"edit_one": edit_one, "create_one": create_one}
        if pieces:
            variants.update(edit_all=edit_all, create_all=create_all)
        times = {k: [] for k in variants}
        for r in range(args.warmup + args.steps):
            for k, fn in variants.items():
                t0 = time.perf_counter()
                fn(r + 1)
                dt = (time.perf_counter() - t0) * 1e3
                if r >= args.warmup:
                    times[k].append(dt)
        frame_only = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            frame(ha)
            frame_only.append((time.perf_counter() - t0) * 1e3)
        res = {k: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v)} for k, v in times.items()}
        res["frame_only"] = {"median_ms": statistics.median(frame_only), "min_ms": min(frame_only), "max_ms": max(frame_only)}
        results["workloads"][wl] = res
        print(json.dumps({"workload": wl, "device": name, "limits": limits, **{k: round(v["median_ms"], 4) for k, v in res.items()}}),
              flush=True)
        api.lib.c2rt_scene_destroy(hb)
        api.lib.c2rt_unpin_host_buffer(argb.ctypes.data)
        a.close()
        b.close()
    c2.shutdown()
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(results, fh, indent=1)


if __name__ == "__main__":
    main()
