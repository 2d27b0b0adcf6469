"""Shaded ray queries against the AA-off colour frame of the same size: the pixel-corner camera rays of C1, C2 and C4 generated
on the device with torch from the frame's camera vectors, shaded by c2rt_shade_rays_device in row order, in 8x4-pixel warp
order and shuffled, next to the colour frame with aa_enabled = 0 (c2rt_render_device, rgb plane only, as the queries), and an
equirectangular panorama from the camera position with the same ray count, row order (no frame can express it).  Device time
per call from CUDA events, the calls alternating step by step, L2 overwritten (untimed) before every timed call.  Prints the
device name, power limit and max SM clock with the numbers, one JSON line per workload.  C1 is for information: its frame
runs on the one-plane kernel, which takes its plane hits from per-row tables, while queries are general rays.

  python profiles/shade_time.py [--steps 10] [--warmup 2] [--out result.json]
"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (scene file, width, height); bench.py's workloads of the same names
    "c1": ("scenes/lecture4-proc-texture.sdl", 1920, 1080),
    "c2": ("scenes/lecture5.sdl", 3840, 2160),
    "c4": ("scenes/chessboard.sdl", 7680, 4320),
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


def camera_rays(torch, cam, w, h, order):
    """Directions upLeft + du x / W + dv y / H - pos of every pixel corner, [h*w, 3] float64 on the device."""
    dev = "cuda"
    pos = torch.tensor(cam.pos[:], dtype=torch.float64, device=dev)
    ul = torch.tensor(cam.up_left[:], dtype=torch.float64, device=dev)
    du = torch.tensor(cam.up_right[:], dtype=torch.float64, device=dev) - ul
    dv = torch.tensor(cam.down_left[:], dtype=torch.float64, device=dev) - ul
    ys, xs = torch.meshgrid(torch.arange(h, device=dev, dtype=torch.float64), torch.arange(w, device=dev, dtype=torch.float64),
                            indexing="ij")
    if order == "patches":   # 32 consecutive queries = one 8x4 pixel patch, as the frame kernels' warps
        ys = ys.reshape(h // 4, 4, w // 8, 8).permute(0, 2, 1, 3)
        xs = xs.reshape(h // 4, 4, w // 8, 8).permute(0, 2, 1, 3)
    x, y = xs.reshape(-1, 1), ys.reshape(-1, 1)
    d = ul + du * (x / w) + dv * (y / h) - pos
    if order == "shuffled":
        g = torch.Generator(device=dev)
        g.manual_seed(1)
        d = d[torch.randperm(len(d), device=dev, generator=g)]
    return pos.expand_as(d).contiguous(), d.contiguous()


def panorama_rays(torch, cam, w, h):
    """Equirectangular panorama from the camera position: pixel centre (x, y) looks at longitude 2 pi (x + 0.5) / w - pi and
    latitude pi / 2 - pi (y + 0.5) / h, y up; row order."""
    dev = "cuda"
    pos = torch.tensor(cam.pos[:], dtype=torch.float64, device=dev)
    ys, xs = torch.meshgrid(torch.arange(h, device=dev, dtype=torch.float64), torch.arange(w, device=dev, dtype=torch.float64),
                            indexing="ij")
    lon = (xs.reshape(-1) + 0.5) * (2 * math.pi / w) - math.pi
    lat = math.pi / 2 - (ys.reshape(-1) + 0.5) * (math.pi / h)
    d = torch.stack([torch.cos(lat) * torch.sin(lon), torch.sin(lat), torch.cos(lat) * torch.cos(lon)], dim=1)
    return pos.expand_as(d).contiguous(), d.contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
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
        st.aa_enabled = 0
        ambient = list(st.ambient_light)
        handle = g.device_scene()
        n = w * h
        cur = torch.cuda.current_stream().cuda_stream
        rays = {k: camera_rays(torch, cam, w, h, k) for k in ("rows", "patches", "shuffled")}
        rays["panorama"] = panorama_rays(torch, cam, w, h)
        frame = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
        rgb = torch.empty((n, 3), dtype=torch.float32, device="cuda")

        def shade(k):
            o, d = rays[k]
            return lambda: api.shade_rays_device(handle, n, o.data_ptr(), d.data_ptr(), ambient, d_rgb=rgb.data_ptr(), stream=cur)
        calls = {
            "colour_frame_aa_off": lambda: api.render_device(handle, cam, st, frame.data_ptr(), None, stream=cur),
            "shade_rows": shade("rows"), "shade_patches": shade("patches"), "shade_shuffled": shade("shuffled"),
            "shade_panorama": shade("panorama"),
        }
        for _ in range(args.warmup):
            for f in calls.values():
                f()
        torch.cuda.synchronize()
        # the row-order colours against the frame they reproduce (the rays here are formed by torch, not the kernel's fma chain)
        calls["shade_rows"]()
        calls["colour_frame_aa_off"]()
        torch.cuda.synchronize()
        diff = (rgb - frame.reshape(-1, 3)).abs().amax(dim=1)
        ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)] for k in calls}
        for i in range(args.steps):
            for k, f in calls.items():
                flush.fill_(1)
                ev[k][i][0].record()
                f()
                ev[k][i][1].record()
        torch.cuda.synchronize()
        line = {"workload": wl, "scene": path, "width": w, "height": h, "rays": n, "steps": args.steps,
                "device": name, "power_limit_max_sm_clock": power,
                "rows_vs_frame_max_abs_diff": float(diff.max().item()), "rows_vs_frame_px_over_1e-5": int((diff > 1e-5).sum().item())}
        for k in calls:
            v = sorted(a.elapsed_time(b) for a, b in ev[k])
            line[f"{k}_ms_median"] = v[len(v) // 2]
            line[f"{k}_ms_min"] = v[0]
            line[f"{k}_ms_max"] = v[-1]
        for k in ("shade_rows", "shade_patches", "shade_shuffled", "shade_panorama"):
            line[f"{k}_over_frame"] = line[f"{k}_ms_median"] / line["colour_frame_aa_off_ms_median"]
        print(json.dumps(line), flush=True)
        results.append(line)
        del rays, frame, rgb
        g.close()
    c2.shutdown()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
