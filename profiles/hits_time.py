"""Hit frame (c2rt_render_hits_device, all four planes) against colour frame (c2rt_render_device, RGB) on the same scene and
camera: device time per frame from CUDA events, the two calls alternating step by step, L2 overwritten (untimed) before every
timed call as bench.py does.  Prints the device name and power limit with the numbers, one JSON line per workload.

  python profiles/hits_time.py [--steps 20] [--warmup 3] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (scene file, width, height); C1, C2 and C4 are bench.py's workloads of the same names
    "c1": ("scenes/lecture4-proc-texture.sdl", 1920, 1080),
    "c2": ("scenes/lecture5.sdl", 3840, 2160),
    "c4": ("scenes/chessboard.sdl", 7680, 4320),
    "nested_1080": ("tests/scenes/nested.sdl", 1920, 1080),
}
L2_FLUSH_BYTES = 256 << 20   # > 126 MB L2


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
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import chess2rt_b200 as c2
    from chess2rt_b200 import api
    name, power = device_info()
    print(f"device: {name}; power limit, max SM clock: {power}", flush=True)
    c2.init(1, [0])
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")
    results = []
    for wl, (path, w, h) in WORKLOADS.items():
        g = c2.HostScene(os.path.join(ROOT, path))
        g.set_frame_size(w, h)
        cam, st = g.frame_blocks(seed=0xC2E55)
        handle = g.device_scene()
        rgb = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
        node = torch.empty((h, w), dtype=torch.int32, device="cuda")
        dist = torch.empty((h, w), dtype=torch.float32, device="cuda")
        normal = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
        uv = torch.empty((h, w, 2), dtype=torch.float32, device="cuda")
        cur = torch.cuda.current_stream().cuda_stream
        calls = {
            "colour": lambda: api.render_device(handle, cam, st, rgb.data_ptr(), None, None, cur),
            "hits": lambda: api.render_hits_device(handle, cam, st, node.data_ptr(), dist.data_ptr(), normal.data_ptr(), uv.data_ptr(),
                                                   stream=cur),
        }
        for _ in range(args.warmup):
            for f in calls.values():
                f()
        torch.cuda.synchronize()
        ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)] for k in calls}
        for i in range(args.steps):
            for k, f in calls.items():
                flush.fill_(1)
                ev[k][i][0].record()
                f()
                ev[k][i][1].record()
        torch.cuda.synchronize()
        ms = {k: sorted(a.elapsed_time(b) for a, b in ev[k]) for k in calls}
        line = {"workload": wl, "scene": path, "width": w, "height": h, "steps": args.steps, "device": name, "power_limit": power}
        for k, v in ms.items():
            line[f"{k}_ms_median"] = v[len(v) // 2]
            line[f"{k}_ms_min"] = v[0]
            line[f"{k}_ms_max"] = v[-1]
        line["hits_over_colour"] = line["hits_ms_median"] / line["colour_ms_median"]
        line["hit_pixels"] = int((node >= 0).sum().item())
        print(json.dumps(line), flush=True)
        results.append(line)
        g.close()
    c2.shutdown()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
