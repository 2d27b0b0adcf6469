"""Partial frames after edits: host wall time from the start of an edit to a synchronised ARGB-only frame, c2rt_render (the whole
frame) against c2rt_render_update (the tiles the edit can have changed; HostScene.render / render_update).  Every repetition
switches between two states, so each edit changes the scene; the two variants alternate within each repetition, each on its
own host scene (the update's cache holds its own buffers).  Medians (min - max) over --steps repetitions after --warmup, with
tiles_rendered / tiles_total of the update.  Prints and records the device name, power limit and max SM clock.

  python profiles/update_time.py [--steps 15] [--warmup 3] [--out profiles/r14_update_time.json]

Workloads: chessboard at 1920x1080, 3840x2160 and 7680x4320, a one-pawn move step (e2 between z -50 and -45) and a highlight
(e2 pointed at black_piece and back); lecture5 at 1920x1080, a sphere moved; a camera orbit step at each chessboard size (every
tile changes: the cost of the full path against c2rt_render).
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from edit_time import device_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import chess2rt_b200 as c2

    if c2.device_count() < 1:
        raise SystemExit("update_time.py needs a CUDA device: libc2rt.so has no CPU fallback")
    c2.init(1, [0])
    chess, lecture5 = os.path.join(ROOT, "scenes", "chessboard.sdl"), os.path.join(ROOT, "scenes", "lecture5.sdl")

    def pawn(s, k):
        s.place_node("e2", translate=(10.0, 0.0, -50.0 + 5.0 * (k % 2)))

    def highlight(s, k):
        s.set_node_shader("e2", "black_piece" if k % 2 == 0 else "white_piece")

    def sphere(s, k):
        s.place_node(3, translate=(100.0, 15.0 + 10.0 * (k % 2), 256.0))

    def orbit(s, k):
        s.camera_rotate(0.5 if k % 2 == 0 else -0.5)

    workloads = []
    for size in ((1920, 1080), (3840, 2160), (7680, 4320)):
        for name, edit in (("pawn_move", pawn), ("highlight", highlight), ("camera_orbit", orbit)):
            workloads.append((f"chessboard_{name}_{size[0]}x{size[1]}", chess, size, edit))
    workloads.append(("lecture5_sphere_move_1920x1080", lecture5, (1920, 1080), sphere))

    results = {"device": device_info(), "steps": args.steps, "warmup": args.warmup, "workloads": {}}
    print(json.dumps(results["device"]))
    for name, path, size, edit in workloads:
        scenes = {}
        for v in ("render", "update"):
            s = c2.HostScene(path)
            s.set_frame_size(*size)
            scenes[v] = s
        out = np.empty((size[1], size[0]), np.uint32)   # render's plane, persistent as render_update's are
        times = {"render": [], "update": []}
        tiles = []
        for k in range(args.warmup + args.steps):
            for v in ("render", "update"):
                s = scenes[v]
                t0 = time.perf_counter()
                edit(s, k)
                if v == "render":
                    s.render(argb_only=True, out_argb=out)
                else:
                    info = s.render_update(argb_only=True)[3]
                t = (time.perf_counter() - t0) * 1e3
                if k >= args.warmup:
                    times[v].append(t)
                    if v == "update":
                        tiles.append((info["tiles_rendered"], info["tiles_total"], info["full"]))
        row = {v: {"median_ms": statistics.median(ts), "min_ms": min(ts), "max_ms": max(ts)} for v, ts in times.items()}
        row["tiles_rendered_median"] = statistics.median(t[0] for t in tiles)
        row["tiles_total"] = tiles[0][1]
        row["full_frames"] = sum(t[2] for t in tiles)
        row["update_over_render"] = row["update"]["median_ms"] / row["render"]["median_ms"]
        results["workloads"][name] = row
        print(f"{name:40s} render {row['render']['median_ms']:8.3f} ms ({row['render']['min_ms']:.3f}-{row['render']['max_ms']:.3f})"
              f"  update {row['update']['median_ms']:8.3f} ms ({row['update']['min_ms']:.3f}-{row['update']['max_ms']:.3f})"
              f"  tiles {row['tiles_rendered_median']:.0f}/{row['tiles_total']}  ratio {row['update_over_render']:.3f}", flush=True)
        for s in scenes.values():
            s.close()
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(results, fh, indent=1)


if __name__ == "__main__":
    main()
