"""Ray queries against the hit frame on the same rays: the camera rays of C2 and C4 generated on the device with torch from
the frame's camera vectors, traced by c2rt_trace_rays_device in row order, in 8x4-pixel warp order and shuffled, next to the
hit frame of the same frame (c2rt_render_hits_device), and c2rt_test_visibility_device from the row-order hit points
(offset by N 1e-6) to light 0.  Device time per call from CUDA events, the calls alternating step by step, L2 overwritten
(untimed) before every timed call.  Prints the device name, power limit and max SM clock with the numbers, one JSON line
per workload.

  python profiles/rays_time.py [--steps 10] [--warmup 2] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (scene file, width, height); bench.py's workloads of the same names
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
        handle = g.device_scene()
        n = w * h
        cur = torch.cuda.current_stream().cuda_stream
        rays = {k: camera_rays(torch, cam, w, h, k) for k in ("rows", "patches", "shuffled")}
        out = {"node": torch.empty(n, dtype=torch.int32, device="cuda"), "dist": torch.empty(n, dtype=torch.float64, device="cuda"),
               "p": torch.empty((n, 3), dtype=torch.float64, device="cuda"), "normal": torch.empty((n, 3), dtype=torch.float64, device="cuda"),
               "uv": torch.empty((n, 2), dtype=torch.float64, device="cuda")}
        hp = {"node": torch.empty((h, w), dtype=torch.int32, device="cuda"), "dist": torch.empty((h, w), device="cuda"),
              "normal": torch.empty((h, w, 3), device="cuda"), "uv": torch.empty((h, w, 2), device="cuda")}
        # visibility queries: the row-order hit points (+ N 1e-6) to light 0
        o, d = rays["rows"]
        api.trace_rays_device(handle, n, o.data_ptr(), d.data_ptr(), *(out[k].data_ptr() for k in ("node", "dist", "p", "normal", "uv")),
                              stream=cur)
        torch.cuda.synchronize()
        hit = out["node"] >= 0
        frm = (out["p"][hit] + out["normal"][hit] * 1e-6).contiguous()
        dsc = g.desc().contents
        light = torch.tensor(dsc.light_pos[0:3], dtype=torch.float64, device="cuda").expand_as(frm).contiguous()
        vis = torch.empty(len(frm), dtype=torch.uint8, device="cuda")
        nv = len(frm)

        def trace(k):
            o, d = rays[k]
            return lambda: api.trace_rays_device(handle, n, o.data_ptr(), d.data_ptr(),
                                                 *(out[q].data_ptr() for q in ("node", "dist", "p", "normal", "uv")), stream=cur)
        calls = {
            "hit_frame": lambda: api.render_hits_device(handle, cam, st, *(hp[q].data_ptr() for q in ("node", "dist", "normal", "uv")),
                                                        stream=cur),
            "rays_rows": trace("rows"), "rays_patches": trace("patches"), "rays_shuffled": trace("shuffled"),
            "visibility_light0": lambda: api.test_visibility_device(handle, nv, frm.data_ptr(), light.data_ptr(), vis.data_ptr(), stream=cur),
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
        line = {"workload": wl, "scene": path, "width": w, "height": h, "rays": n, "visibility_queries": nv, "steps": args.steps,
                "device": name, "power_limit_max_sm_clock": power}
        for k in calls:
            v = sorted(a.elapsed_time(b) for a, b in ev[k])
            line[f"{k}_ms_median"] = v[len(v) // 2]
            line[f"{k}_ms_min"] = v[0]
            line[f"{k}_ms_max"] = v[-1]
        for k in ("rays_rows", "rays_patches", "rays_shuffled"):
            line[f"{k}_over_hit_frame"] = line[f"{k}_ms_median"] / line["hit_frame_ms_median"]
        line["hit_rays"] = int(hit.sum().item())
        line["visible"] = int(vis.sum().item())
        print(json.dumps(line), flush=True)
        results.append(line)
        del rays, out, hp, frm, light, vis
        g.close()
    c2.shutdown()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
