#!/usr/bin/env python
"""bench.py — the headline benchmark of BASELINE.json: Mrays/s and frames/s at 1920x1080.

A "step" is ONE FRAME of the workload rendered by the hot path.  At N=1 the workload is
BASELINE.json configs[1]: data/lecture4-proc-texture.sdl at 1920x1080 (procedural texture + Lambert +
shadow rays, 5 samples per pixel).  With N>1 ranks (one process per GPU, torchrun) the same frame is
split into interleaved 8-row bands, each rank renders its bands, and the bands are gathered to rank 0
(`--gather p2p`, the default: kernels store straight into rank 0's frame through a CUDA-IPC mapping over
NVLink, completion is signalled inside the render kernel and the ranks start each frame through a
device-side gate; `--gather nccl`: NCCL gather + the library's scatter kernel); total work is fixed, so
scaling is "strong".

  value      device-resident throughput: inputs (scene, camera) already on the GPU, output left in HBM
  e2e        the same metric through the public host API (c2rt_render via the host mirror) with HOST
             buffers: camera/settings go down as launch parameters, the float frame comes back to
             pinned host memory inside the timed region
  roofline   FP32 CUDA-core roofline (the path is FMA-bound, not HBM- or tensor-bound: DESIGN.md §4):
             achieved = algorithmic FLOPs of the frame (counted by the oracle's counting scalar,
             chess2rt_b200/workloads.json) / mean kernel time (CUDA events)
  cpu_baseline  the CPU oracle (C++ restatement of the reference: the D reference cannot be built in
             this image) timed on the box's host cores on the same frame
  parity     (N = 1, with the CPU leg) the frame the e2e leg delivered against the oracle: max |diff|, pixels over 1e-3, share
             of 8-bit pixels off by > 1 LSB, a diff image under gpurun_out/ when that directory exists; the run fails above the
             bar.  Each scaling target carries the same check on 96 rows of its frame
  scaling_targets  BASELINE.json configs[2..4] (lecture5 4K, zaphod 4K DOF, chessboard 8K) measured in the same run
             at the same N: ms per frame, efficiency against rank 0 rendering the frame alone, frame check
`--impl reference` times that CPU implementation alone with the same metric/config.
`--workload` picks another configuration (c0..c4, chess1080, chess4k); the default is the headline one.
`--dump-outputs DIR` writes the frame the last timed step rendered as DIR/frame.npy (float32 [H, W, 3], what a caller of
c2rt_render_device receives); inputs are fixed (scene file, camera, RNG seed), so two builds can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (scene file, width, height, overrides)
    "c0": ("scenes/lecture4.sdl", 640, 480, {}),
    "c1": ("scenes/lecture4-proc-texture.sdl", 1920, 1080, {}),
    "c2": ("scenes/lecture5.sdl", 3840, 2160, {}),
    "c3": ("scenes/zaphod-sky.sdl", 3840, 2160, {}),      # configs[3]: zaphod.sdl + the cubemap-environment extension (DESIGN.md; SURVEY.md F3)
    "c3_nosky": ("scenes/zaphod.sdl", 3840, 2160, {}),   # the scene file as the reference ships it (same frame: no ray of it misses)
    "c4": ("scenes/chessboard.sdl", 7680, 4320, {}),
    "chess1080": ("scenes/chessboard.sdl", 1920, 1080, {}),
    "chess4k": ("scenes/chessboard.sdl", 3840, 2160, {}),
    "lecture5_1080": ("scenes/lecture5.sdl", 1920, 1080, {}),
}
DEFAULT_WORKLOAD = "c1"
SCALING_TARGETS = ["c2", "c3", "c4"]   # BASELINE.json configs[2], [3], [4]


def workload_label(name):
    """config.workload: the same string in both arms (ours and --impl reference)."""
    path, w, h, _ = WORKLOADS[name]
    return "%s: %s at %dx%d" % (name, path, w, h)
BAND_ROWS = 8
RNG_SEED = 0xC2E55
L2_FLUSH_BYTES = 256 << 20  # > 126 MB L2
DUMP_BYTES = 64 << 20       # --dump-outputs writes at most this much


def dump_frame(out_dir, frame):
    """--dump-outputs: `frame` ([H, W, 3] float32) as out_dir/frame.npy.  A frame larger than DUMP_BYTES (the 8K workload) keeps
    every k-th row from row 0, the smallest k that fits, and out_dir/frame_rows.npy lists the rows kept."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    frame = np.ascontiguousarray(frame, dtype=np.float32)
    H = frame.shape[0]
    if frame.nbytes > DUMP_BYTES:
        fit = (DUMP_BYTES - 8 * H - 4096) // frame[0].nbytes   # room for the row list and the two .npy headers
        rows = np.arange(0, H, -(-H // fit))
        frame = frame[rows]
        np.save(os.path.join(out_dir, "frame_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "frame.npy"), frame)


def load_calibration():
    p = os.path.join(ROOT, "chess2rt_b200", "workloads.json")
    return json.load(open(p)) if os.path.exists(p) else {}


def calibrate(names):
    """Counts algorithmic FLOPs and rays of each workload with the oracle's counting build (CPU, slow)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_binding import OracleScene
    cal = load_calibration()
    for name in names:
        path, w, h, over = WORKLOADS[name]
        s = OracleScene(os.path.join(ROOT, path), count_flops=True)
        s.set_frame_size(w, h)
        s.override(**over)
        if name in ("c3", "c4"):
            # exact counts for 8K / DOF frames take CPU-minutes: count every 16th 8-row band and scale
            tot = {"flops": 0, "primary": 0, "shadow": 0}
            rows = 0
            for y0 in range(0, h, 8 * 16):
                _, st = s.render_rows(y0, min(h, y0 + 8), seed=RNG_SEED)
                tot["flops"] += st.flops; tot["primary"] += st.primary_rays; tot["shadow"] += st.shadow_rays
                rows += min(h, y0 + 8) - y0
            k = h / rows
            cal[name] = {"scene": path, "width": w, "height": h, "flops": int(tot["flops"] * k),
                         "primary_rays": int(tot["primary"] * k), "shadow_rays": int(tot["shadow"] * k),
                         "exact": False, "how": "every 16th 8-row band counted, scaled by rows"}
        else:
            _, st = s.render(seed=RNG_SEED)
            cal[name] = {"scene": path, "width": w, "height": h, "flops": int(st.flops), "primary_rays": int(st.primary_rays),
                         "shadow_rays": int(st.shadow_rays), "exact": True, "how": "full frame, oracle counting scalar"}
        print(name, cal[name], flush=True)
    json.dump(cal, open(os.path.join(ROOT, "chess2rt_b200", "workloads.json"), "w"), indent=1, sort_keys=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_frame_seconds(path, w, h, over, threads, min_seconds=2.0, max_frames=5):
    """Times the CPU oracle on full frames of the workload (bounded: stops after min_seconds or max_frames)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_binding import OracleScene
    s = OracleScene(os.path.join(ROOT, path))
    s.set_frame_size(w, h)
    s.override(**over)
    times, rays = [], None
    t_all = time.perf_counter()
    while len(times) < max_frames and (time.perf_counter() - t_all < min_seconds or not times):
        _, st = s.render(threads=threads, seed=RNG_SEED)
        times.append(st.seconds)
        rays = st.primary_rays + st.shadow_rays
    return times, rays


def cpu_rows_seconds(path, w, h, over, threads, rows):
    """Bounded sample for frames too big to render whole on the CPU: `rows` rows spread over the frame."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_binding import OracleScene
    s = OracleScene(os.path.join(ROOT, path))
    s.set_frame_size(w, h)
    s.override(**over)
    sec, rays, done = 0.0, 0, 0
    n_win = max(1, rows // 8)
    for i in range(n_win):
        y0 = min(h - 8, (h // n_win) * i) // 8 * 8
        _, st = s.render_rows(y0, min(h, y0 + 8), threads=threads, seed=RNG_SEED)
        sec += st.seconds; rays += st.primary_rays + st.shadow_rays; done += min(h, y0 + 8) - y0
    return sec, rays, done


def oracle_parity(path, w, h, over, gpu_rows, rows=None, diff_path=None):
    """Parity check alongside timing (SURVEY.md section 8(d); untimed, rank 0, N = 1, part of the CPU leg): the frame the product
    path rendered for this workload against the CPU oracle — max |diff|, pixels over 1e-3, share of 8-bit pixels off by more than
    1 LSB; the run FAILS above the bar.  `gpu_rows(y0, y1)` returns rows [y0, y1) of the GPU frame as a numpy array.
    rows=None: the whole frame; otherwise `rows` rows in windows of 8 spread over the frame (bounded CPU time for 4K / 8K frames).
    diff_path: the per-pixel max |diff| as an 8-bit PGM, 255 = 1e-3 (whole-frame checks only)."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_binding import OracleScene, parity_report
    o = OracleScene(os.path.join(ROOT, path))
    o.set_frame_size(w, h)
    o.override(**over)
    threads = os.cpu_count() or 1
    if rows is None:
        wins = [(0, h)]
    else:
        n_win = max(1, rows // 8)
        wins = sorted({min(h - 8, (h // n_win) * i) // 8 * 8 for i in range(n_win)})
        wins = [(y0, min(h, y0 + 8)) for y0 in wins]
    got, ref = [], []
    for y0, y1 in wins:
        r, _ = o.render_rows(y0, y1, threads=threads, seed=RNG_SEED)
        ref.append(r)
        got.append(np.asarray(gpu_rows(y0, y1), dtype=np.float32))
    got, ref = np.concatenate(got), np.concatenate(ref)
    rep = parity_report(got, ref)
    rep["sample"] = "whole frame" if rows is None else "%d rows (windows of 8 rows spread over the frame)" % got.shape[0]
    rep["bar"] = "0 px over 1e-3 absolute; <= 0.1 % of 8-bit pixels off by more than 1 LSB"
    rep["pass"] = rep["px_over_1e-3"] == 0 and rep["frac_over_1lsb"] <= 1e-3
    if diff_path and rows is None:
        d = np.abs(got.astype(np.float64) - ref.astype(np.float64)).max(axis=-1)
        img = np.clip(d / 1e-3 * 255.0, 0, 255).astype(np.uint8)
        with open(diff_path, "wb") as f:
            f.write(b"P5\n%d %d\n255\n" % (w, h))
            f.write(img.tobytes())
        rep["diff_image"] = os.path.relpath(diff_path, ROOT) + " (max |diff| per pixel, 255 = 1e-3)"
    return rep


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (the C++ oracle port; the D
    original needs dmd/ldc2 + dub + gfm + sdlang-d, none present: DESIGN.md) on all host cores."""
    if rank != 0:
        return
    path, w, h, over = WORKLOADS[args.workload]
    threads = os.cpu_count() or 1
    big = w * h > 3840 * 2160 or args.workload == "c3"
    step_s, rays = [], None
    sample = "full frame per step"
    for i in range(args.warmup + args.steps):
        if big:
            sec, r, done = cpu_rows_seconds(path, w, h, over, threads, rows=64)
            sec, r = sec * h / done, r * h / done
            sample = "64 rows (8 windows of 8 rows spread over the frame) per step, scaled to the frame"
        else:
            t, r = cpu_frame_seconds(path, w, h, over, threads, min_seconds=0, max_frames=1)
            sec = t[0]
        if i >= args.warmup:
            step_s.append(sec)
        rays = r
    ms = 1e3 * sum(step_s) / len(step_s)
    val = rays / (ms * 1e-3) / 1e6
    line = {
        "impl": "reference", "metric": "Mrays/s at %dx%d" % (w, h), "value": val, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "frames_per_s": 1e3 / ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64 geometry / f32 colour", "data": "synthetic (bundled scene file, no external data)",
        "config": {"workload": workload_label(args.workload), "rays_per_frame": rays},
        "cpu_baseline": {"value": val, "unit": "Mrays/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--gather", default="auto", choices=["auto", "nccl", "p2p"])
    ap.add_argument("--calibrate", nargs="*", default=None, help="(CPU) recount algorithmic FLOPs/rays of the named workloads")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-scaling-target", action="store_true", help="skip the side measurement of the 8K chessboard scene")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the frame of the last timed step as DIR/frame.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.calibrate is not None:
        calibrate(args.calibrate or ["c0", "c1", "c2", "chess1080"])
        return

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import chess2rt_b200 as c2
    from chess2rt_b200 import api, bands

    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    torch.cuda.set_device(local_rank)
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")  # host-side waits that must not occupy a GPU (see the e2e leg)
    c2.init(1, [local_rank])
    stream = torch.cuda.current_stream().cuda_stream
    flush_buf = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    class DeviceRun:
        """One workload set up for device-resident stepping on this rank: scene upload, band, output buffers, gather."""

        def __init__(self, name, gather):
            import ctypes as C
            self.name = name
            self.path, self.W, self.H, self.over = WORKLOADS[name]
            W, H = self.W, self.H
            self.scene = c2.HostScene(os.path.join(ROOT, self.path))
            self.scene.set_frame_size(W, H)
            self.scene.override(**self.over)
            self.handle = self.scene.device_scene()
            self.cam, self.st = self.scene.frame_blocks(seed=RNG_SEED)
            self.launches = 0
            self.peer_frame_ptr = None
            self.frame = None
            self.pad = bands.rows_padded(H, world, BAND_ROWS)
            if world == 1:
                self.mode = "none"
                self.band = None
                self.frame = torch.empty((H, W, 3), dtype=torch.float32, device="cuda")
                self.out_ptr = self.frame.data_ptr()
                return
            self.mode = "nccl" if gather == "nccl" else "p2p"
            if self.mode == "p2p":
                # rank 0 owns the frame; every other rank maps it (CUDA IPC) and its kernel stores bands into it over NVLink
                ok = 1
                handle_bytes = [None]
                try:
                    if rank == 0:
                        p = C.c_void_p()
                        api._check(api.lib.c2rt_frame_alloc(H * W * 12 + 256, C.byref(p)))   # frame + completion flags
                        hb = (C.c_uint8 * 64)()
                        api._check(api.lib.c2rt_frame_export(p, hb))
                        handle_bytes = [bytes(hb)]
                        self.peer_frame_ptr = p.value
                except Exception:
                    ok = 0
                dist.broadcast_object_list(handle_bytes, src=0)
                if rank != 0 and handle_bytes[0] is not None:
                    try:
                        hb = (C.c_uint8 * 64).from_buffer_copy(handle_bytes[0])
                        p = C.c_void_p()
                        api._check(api.lib.c2rt_frame_import(hb, C.byref(p)))
                        self.peer_frame_ptr = p.value
                    except Exception:
                        ok = 0
                okt = torch.tensor([ok if handle_bytes[0] is not None else 0], device="cuda")
                dist.all_reduce(okt, op=dist.ReduceOp.MIN)
                if int(okt[0]) == 0:
                    if gather == "p2p":
                        raise SystemExit("--gather p2p: CUDA IPC mapping of rank 0's frame failed")
                    self.mode = "nccl"   # auto: fall back to the NCCL gather
            if self.mode == "p2p":
                # uint32 flags[world + 1] behind the frame, in rank 0's memory: [0] start-gate counter, [r] last frame rank r
                # completed, [world] time-outs (c2rt.h c2rt_band.done_flags, c2rt_gate)
                self.flags_ptr = self.peer_frame_ptr + H * W * 12
                self.band = api.Band(rank, world, BAND_ROWS, 0, self.flags_ptr, 0, 0)
                self.out_ptr = self.peer_frame_ptr
                if os.environ.get("C2RT_DIAG_LOCAL_PEER_STORES") == "1" and rank != 0:
                    # DIAGNOSTIC ONLY (the gathered frame is then wrong and verify() is skipped): peers store their bands into a
                    # local frame instead of rank 0's, everything else unchanged — what do the NVLink stores cost the peer kernels?
                    self.local_frame = torch.empty((H, W, 3), dtype=torch.float32, device="cuda")
                    self.out_ptr = self.local_frame.data_ptr()
                self.frame_no = 0
                dist.barrier()   # c2rt_frame_alloc zero-fills: the flags start at 0 before any rank signals
            else:
                self.band = api.Band(rank, world, BAND_ROWS, 1, None, 0, 0)
                self.mine = torch.empty((self.pad, W, 3), dtype=torch.float32, device="cuda")
                self.gathered = torch.empty((world, self.pad, W, 3), dtype=torch.float32, device="cuda") if rank == 0 else None
                self.frame = torch.empty((H, W, 3), dtype=torch.float32, device="cuda") if rank == 0 else None
                self.out_ptr = self.mine.data_ptr()

        def step(self, cam=None, st=None):
            """One frame on this rank's stream: [start gate] render [gather].  With p2p the gather IS the render kernel: peers
            store their bands into rank 0's frame and raise their flag from a one-thread kernel behind it, the last CTA of
            rank 0's kernel waits for all flags (c2rt.h c2rt_band.done_flags)."""
            cur = torch.cuda.current_stream().cuda_stream
            if self.mode == "p2p":
                self.frame_no += 1
                api._check(api.lib.c2rt_gate(self.flags_ptr, world, self.frame_no, cur))   # (one gate per frame: round == frame number)
                self.band.frame_no = self.frame_no
                self.launches += 1
            c2.render_device(self.handle, cam or self.cam, st or self.st, self.out_ptr, None, self.band, cur)
            self.launches += 2 if (self.mode == "p2p" and rank != 0) else 1   # peers: render kernel + the one-thread flag kernel
            if self.mode == "nccl":
                dist.gather(self.mine, list(self.gathered.unbind(0)) if rank == 0 else None, dst=0)
                if rank == 0:
                    c2.deinterleave(self.gathered.data_ptr(), self.frame.data_ptr(), self.W, self.H, 3, world, BAND_ROWS, self.pad, cur)
                    self.launches += 1

        def timeouts(self):
            """flags[world]: gate / completion waits that gave up (a rank died or never arrived).  Must be 0."""
            if self.mode != "p2p":
                return 0
            import ctypes as C
            t = torch.zeros(1, dtype=torch.int32, device="cuda")
            if rank == 0:
                got = torch.zeros(1, dtype=torch.int32).pin_memory()
                api._check(api.lib.c2rt_frame_download(got.data_ptr(), C.c_void_p(self.flags_ptr + 4 * world), 4, torch.cuda.current_stream().cuda_stream))
                torch.cuda.synchronize()
                t[0] = int(got[0])
            dist.broadcast(t, src=0)
            return int(t[0])

        def count_rays(self):
            cam_c, st_c = self.scene.frame_blocks(seed=RNG_SEED, count_rays=True)
            self.step(cam_c, st_c)
            prim, shad = c2.read_ray_counters(self.handle, stream)
            counts = torch.tensor([prim, shad], dtype=torch.int64, device="cuda")
            if world > 1:
                dist.all_reduce(counts)
            return int(counts[0]), int(counts[1])

        def time_steps(self, steps, warmup):
            """EXACTLY `steps` timed frames; L2 flushed between them (untimed); per-step CUDA events; max over ranks.
            Each step is enqueued behind its (untimed) L2-flush kernel, so the host's launch latency is hidden and the
            events bracket device work only; with N > 1 the device-side gate lines the ranks up right before e0.
            Returns (ms per step, launches in the timed region)."""
            for _ in range(warmup):
                flush_buf.fill_(1)
                self.step()
            barrier()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            self.launches = 0
            barrier()
            cur = torch.cuda.current_stream().cuda_stream
            for e0, e1 in ev:
                flush_buf.fill_(1)
                if self.mode == "p2p":
                    # gate in front of e0: waiting for the slowest rank's flush is not frame time
                    self.frame_no += 1
                    api._check(api.lib.c2rt_gate(self.flags_ptr, world, self.frame_no, cur))
                    self.band.frame_no = self.frame_no
                    e0.record()
                    c2.render_device(self.handle, self.cam, self.st, self.out_ptr, None, self.band, cur)
                    self.launches += 2 if rank != 0 else 1   # peers: render kernel + the one-thread flag kernel
                elif self.mode == "nccl":
                    dist.barrier()
                    e0.record()
                    self.step()
                else:
                    e0.record()
                    self.step()
                e1.record()
            barrier()
            t = torch.tensor([sum(e0.elapsed_time(e1) for e0, e1 in ev)], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            n_to = self.timeouts() if world > 1 else 0
            if n_to:
                raise SystemExit(f"{self.name}: {n_to} gate / frame-complete wait(s) timed out: the timed frames are not complete frames")
            return float(t[0]) / steps, self.launches

        def frame_host(self):
            """(rank 0) the frame the last step left in HBM, copied to the host as [H, W, 3] float32."""
            if self.mode == "p2p":
                import ctypes as C
                got = torch.empty((self.H, self.W, 3), dtype=torch.float32, pin_memory=True)
                api._check(api.lib.c2rt_frame_download(got.data_ptr(), C.c_void_p(self.peer_frame_ptr), self.H * self.W * 12,
                                                       torch.cuda.current_stream().cuda_stream))
                torch.cuda.synchronize()
                return got.numpy()
            return self.frame.cpu().numpy()

        def time_alone(self, steps, warmup=2):
            """(N > 1) rank 0 renders the whole frame alone, the other ranks idle: the T(1) of the efficiency figure, same run."""
            ms = 0.0
            if rank == 0:
                alone = torch.empty((self.H, self.W, 3), dtype=torch.float32, device="cuda")
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
                cur = torch.cuda.current_stream().cuda_stream
                for _ in range(warmup):
                    c2.render_device(self.handle, self.cam, self.st, alone.data_ptr(), None, None, cur)
                for e0, e1 in ev:
                    flush_buf.fill_(1)
                    e0.record()
                    c2.render_device(self.handle, self.cam, self.st, alone.data_ptr(), None, None, cur)
                    e1.record()
                torch.cuda.synchronize()
                ms = sum(e0.elapsed_time(e1) for e0, e1 in ev) / steps
                del alone
            if world > 1:
                dist.barrier(group=cpu_group)   # (not an NCCL barrier: its kernel would spin on the idle GPUs' SMs)
            return ms

        def verify(self):
            """(untimed) rank 0: the frame assembled from all ranks' bands equals, bit for bit, the same frame rendered by
            rank 0 alone.  The shared frame is filled with NaNs first, so a band that did not arrive cannot pass for the one a
            previous frame left there."""
            if world == 1:
                return None
            if os.environ.get("C2RT_DIAG_LOCAL_PEER_STORES") == "1":
                return "SKIPPED (C2RT_DIAG_LOCAL_PEER_STORES=1: diagnostic run, the frame is not gathered)"
            import ctypes as C
            cur = torch.cuda.current_stream().cuda_stream
            if self.mode == "p2p" and rank == 0:
                api._check(api.lib.c2rt_frame_memset(C.c_void_p(self.peer_frame_ptr), 0xFF, self.H * self.W * 12, cur))
            elif self.mode == "nccl" and rank == 0:
                self.frame.fill_(float("nan"))
            self.step()   # (p2p: the gate inside keeps the peers' stores behind rank 0's memset)
            W, H = self.W, self.H
            got = None
            if self.mode == "p2p" and rank == 0:
                # the copy-out is enqueued straight behind rank 0's render kernel, BEFORE any host barrier: the end of that kernel
                # alone must mean that every peer's band has arrived
                got = torch.empty((H, W, 3), dtype=torch.float32, pin_memory=True)
                api._check(api.lib.c2rt_frame_download(got.data_ptr(), self.peer_frame_ptr, H * W * 12, cur))
            barrier()
            n_to = self.timeouts()
            if rank != 0:
                return None
            alone = torch.empty((H, W, 3), dtype=torch.float32, device="cuda")
            c2.render_device(self.handle, self.cam, self.st, alone.data_ptr(), None, None, cur)
            if self.mode == "p2p":
                torch.cuda.synchronize()
                same = bool(torch.equal(got, alone.cpu()))
            else:
                torch.cuda.synchronize()
                same = bool(torch.equal(self.frame, alone))
            if n_to:
                return "MISMATCH (%d wait time-outs)" % n_to
            return "bit-identical to the frame rendered by rank 0 alone (shared frame NaN-filled first)" if same else "MISMATCH"

        def close(self):
            import ctypes as C
            if self.peer_frame_ptr:
                if rank == 0:
                    api.lib.c2rt_frame_free(C.c_void_p(self.peer_frame_ptr))
                else:
                    api.lib.c2rt_frame_unimport(C.c_void_p(self.peer_frame_ptr))
            self.scene.close()

    path, W, H, over = WORKLOADS[args.workload]
    run = DeviceRun(args.workload, args.gather)
    gather_mode = run.mode

    # ---- sanity: the workload is the calibrated one (ray counts must match the oracle's) ---------
    cal = load_calibration().get(args.workload)
    prim, shad = run.count_rays()
    if cal and cal.get("exact") and (prim, shad) != (cal["primary_rays"], cal["shadow_rays"]):
        raise SystemExit(f"ray counts {prim}+{shad} differ from the calibrated workload {cal['primary_rays']}+{cal['shadow_rays']}")
    rays_per_frame = prim + shad
    flops_per_frame = cal["flops"] if cal else None

    # ---- roofline denominators: measured on this device before anything is timed -------------------
    peak_tf, peak_mhz = c2.measure_fma_peak(False)
    peak64_tf, _ = c2.measure_fma_peak(True)
    sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
    peaks = {"fp32_tflops": peak_tf, "fp64_tflops": peak64_tf, "sm_mhz_effective": peak_mhz, "sms": sms}

    # ---- timed region ------------------------------------------------------------------------------
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler is not None:
        sampler.start()   # sampled from before the warm-up to the end of the e2e leg (a 1080p frame takes 0.16 ms:
                          # the timed loops alone are shorter than one nvidia-smi period)
    ms_per_step, n_launches = run.time_steps(args.steps, args.warmup)
    kernel_ms = ms_per_step   # one render kernel per rank and step is the whole step (N > 1: it also carries the band gather)
    if args.dump_outputs and rank == 0:
        dump_frame(args.dump_outputs, run.frame_host())

    frame_check = run.verify()
    if world > 1:
        dist.barrier()
    if frame_check and frame_check.startswith("MISMATCH"):
        raise SystemExit("multi-GPU frame differs from the single-GPU frame: " + frame_check)

    # ---- BASELINE.json configs[2..4] beside the headline workload: lecture5 4K, zaphod 4K DOF, chessboard 8K at this N ----
    scaling_targets = []
    if args.workload == DEFAULT_WORKLOAD and not args.no_scaling_target:
        for name in SCALING_TARGETS:
            rn = DeviceRun(name, args.gather)
            pn, sn = rn.count_rays()
            k = max(3, args.steps // 4)
            ms_n, _ = rn.time_steps(k, 3)
            check_n = rn.verify()
            if check_n and check_n.startswith("MISMATCH"):
                raise SystemExit(f"{name}: multi-GPU frame differs from the single-GPU frame: {check_n}")
            ms_1 = rn.time_alone(k) if world > 1 else ms_n
            cal_n = load_calibration().get(name) or {}
            ex_n = executed_fractions(name, ms_1, peaks) if rank == 0 else None
            par_n = None
            if world == 1 and not args.no_cpu_baseline:
                pth_n, w_n, h_n, over_n = WORKLOADS[name]
                par_n = oracle_parity(pth_n, w_n, h_n, over_n, lambda y0, y1: rn.frame[y0:y1].cpu().numpy(), rows=96)
                if not par_n["pass"]:
                    raise SystemExit(f"{name}: the timed frame is not in parity with the oracle: {par_n}")
            scaling_targets.append({
                "workload": workload_label(name), "n_gpus": world, "ms_per_step": ms_n, "ms_per_step_1gpu_same_run": ms_1,
                "efficiency": ms_1 / (world * ms_n), "value": (pn + sn) / (ms_n * 1e-3) / 1e6, "unit": "Mrays/s",
                "frames_per_s": 1e3 / ms_n, "steps": k, "gather": rn.mode, "frame_check": check_n,
                "algorithmic_flops_per_frame": cal_n.get("flops"),
                "achieved_tflops_per_gpu": (cal_n["flops"] / world / (ms_n * 1e-3) / 1e12) if cal_n.get("flops") else None,
                "executed_1gpu": ex_n, "parity": par_n})
            rn.close()

    # ---- e2e: public host API, HOST buffers, copies inside the timed region ------------------------
    pinned = torch.empty((H, W, 3), dtype=torch.float32, pin_memory=True) if rank == 0 else None
    e2e_ms = []
    scene = run.scene
    if world == 1:
        out_np = pinned.numpy()
        for i in range(args.warmup + args.steps):
            flush_buf.fill_(1)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            scene.render(seed=RNG_SEED, out=out_np)      # c2rt_render: launch params down, kernel, frame D2H, sync
            t1 = time.perf_counter()
            if i >= args.warmup:
                e2e_ms.append((t1 - t0) * 1e3)
    else:
        # N > 1: the public host API drives all N devices from ONE process (what the D host does:
        # c2rt_init(N) once, then c2rt_render per frame).  Rank 0 makes those calls; the other ranks wait.
        barrier()
        if rank == 0:
            c2.init(world, list(range(world)))
            scene_n = c2.HostScene(os.path.join(ROOT, path))
            scene_n.set_frame_size(W, H)
            scene_n.override(**over)
            out_np = pinned.numpy()
            for i in range(args.warmup + args.steps):
                t0 = time.perf_counter()
                scene_n.render(seed=RNG_SEED, out=out_np)
                t1 = time.perf_counter()
                if i >= args.warmup:
                    e2e_ms.append((t1 - t0) * 1e3)
            scene_n.close()
        else:
            e2e_ms = [0.0]
        # the waiting ranks must not sit in an NCCL barrier: its kernel would time-slice with rank 0's work on their GPU
        dist.barrier(group=cpu_group)
    e2e_ms_mean = sum(e2e_ms) / len(e2e_ms)

    # ---- the interactive loop (SURVEY.md section 8f-2): the camera turns before every frame (Camera.rotate, what the arrow keys
    # do), the scene stays resident, only the camera / settings blocks go down and only the packed ARGB plane comes back
    interactive = None
    if world == 1:
        import numpy as np
        argb_pinned = torch.empty((H, W), dtype=torch.int32, pin_memory=True)
        a_np = argb_pinned.numpy().view(np.uint32)
        ts = []
        for i in range(args.warmup + args.steps):
            scene.camera_rotate(0.5)
            t0 = time.perf_counter()
            scene.render(seed=RNG_SEED, out_argb=a_np, argb_only=True)
            t1 = time.perf_counter()
            if i >= args.warmup:
                ts.append((t1 - t0) * 1e3)
        scene.camera_rotate(-0.5 * (args.warmup + args.steps))
        interactive = {"ms_per_frame": sum(ts) / len(ts), "frames_per_s": 1e3 * len(ts) / sum(ts), "d2h_bytes_per_frame": W * H * 4,
                       "h2d_bytes_per_frame": C_sizeof_frame_blocks(api),
                       "how": "camera yaw changed before every frame; c2rt_render with rgb == NULL (ARGB-only delivery into a pinned plane)"}
    clocks = sampler.stop() if rank == 0 else None

    if rank == 0:
        value = rays_per_frame / (ms_per_step * 1e-3) / 1e6
        peaks_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
        mp = json.load(open(peaks_file)) if os.path.exists(peaks_file) else {}
        nominal_tf = 2 * 128 * sms * mp.get("sm_max_mhz", 1965.0) * 1e6 / 1e12
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get(args.workload)
        roofline = None
        if flops_per_frame:
            achieved = flops_per_frame / world / (kernel_ms * 1e-3) / 1e12  # per GPU: each renders 1/N of the frame
            roofline = {
                "bound": "fp32", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                "traffic": traffic, "peak_source": "FFMA micro-benchmark measured in this run (c2rt_measure_fma_peak)",
                "peak_nominal": nominal_tf, "frac_nominal": achieved / nominal_tf, "fp64_peak_measured": peak64_tf,
                "algorithmic_flops_per_frame": flops_per_frame, "kernel_ms": kernel_ms,
                "note": "achieved = ALGORITHMIC FLOPs of the reference's arithmetic (oracle counting scalar) / kernel time; culled and "
                        "simplified work still counts, so frac can exceed 1 on many-node scenes.  What the hardware executed is in `executed`",
                "executed": executed_fractions(args.workload, kernel_ms, peaks) if world == 1 else None,
                "hbm": {"achieved": W * H * 12 / world / (kernel_ms * 1e-3) / 1e9, "peak": mp.get("hbm_gbs"), "unit": "GB/s",
                        "note": "framebuffer bytes written per kernel; far below the HBM roof, the kernel is FMA-bound"},
            }
        ingest = None
        if world > 1:
            nb = (world - 1) * W * H * 12 // world
            ingest = {"nvlink_ingest_bytes_per_frame": nb, "floor_ms_at_900GBs": nb / 900e9 * 1e3,
                      "note": "bytes the peers store into rank 0's frame per frame; rank 0's NVLink ingest bounds the gathered frame"}
        line = {
            "metric": "Mrays/s at %dx%d" % (W, H), "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "frames_per_s": 1e3 / ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64 geometry / f32 colour (as the reference)",
            "data": "synthetic (bundled scene file rendered from a fixed camera; no external data)",
            "config": {"workload": workload_label(args.workload), "samples_per_px": prim // (W * H),
                       "rays_per_frame": rays_per_frame, "primary_rays": prim, "shadow_rays": shad,
                       "l2": "flushed between timed steps (256 MiB fill, untimed); per-step CUDA events summed",
                       "parallelism": "row bands of %d rows, interleaved over %d GPU(s), gather=%s" % (BAND_ROWS, world, gather_mode),
                       "launch": "one render kernel per rank and step" + (" (+ a one-thread start gate in front of the timed region; peers raise a flag from a one-thread kernel, rank 0 waits for the flags inside its render kernel)" if gather_mode == "p2p" else ""),
                       "timing": "each step enqueued behind its untimed L2-flush kernel; CUDA events around the step; max over ranks"},
            "roofline": roofline,
            "e2e": {"value": rays_per_frame / (e2e_ms_mean * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_step": e2e_ms_mean,
                    "frames_per_s": 1e3 / e2e_ms_mean, "h2d_bytes_per_step": C_sizeof_frame_blocks(api) * world, "d2h_bytes_per_step": W * H * 12,
                    "how": "host mirror Renderer.renderRT -> c2rt_render into a pinned host frame; " +
                           ("one device, chunked launches with the copy overlapped" if world == 1 else
                            "one process driving %d devices (c2rt_init(%d)), each device copies its own bands to the host" % (world, world))},
            "gpu_launches": n_launches,
            "clocks": clocks,
            "scaling_targets": scaling_targets,
            "multi_gpu_frame_check": frame_check,
            "nvlink": ingest,
            "interactive": interactive,
        }
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            if W * H <= 3840 * 2160 and args.workload != "c3":
                times, rays = cpu_frame_seconds(path, W, H, over, threads, min_seconds=3.0, max_frames=5)
                sec = min(times)
                sample = "%d full frame(s) of the workload, best of" % len(times)
            else:
                s_, rays_, done = cpu_rows_seconds(path, W, H, over, threads, rows=128)
                sec, rays = s_ * H / done, rays_ * H / done
                sample = "128 rows (16 windows of 8 rows spread over the frame), scaled to the frame"
            # one thread beside it (comparable with the reference's published single-thread numbers, perf-results.md:21):
            # 96 rows spread over the frame, scaled
            s1, r1, done1 = cpu_rows_seconds(path, W, H, over, 1, rows=96)
            # parity of the timed workload alongside its timing: the frame the e2e leg just delivered through the public host API
            # against the oracle (whole frame up to 4K without DOF, else 128 rows)
            diff_path = os.path.join(ROOT, "gpurun_out", "bench_parity_diff_%s.pgm" % args.workload) if os.path.isdir(os.path.join(ROOT, "gpurun_out")) else None
            whole = W * H <= 3840 * 2160 and args.workload not in ("c3", "c3_nosky")
            line["parity"] = oracle_parity(path, W, H, over, lambda y0, y1: pinned.numpy()[y0:y1], rows=None if whole else 128, diff_path=diff_path)
            if not line["parity"]["pass"]:
                raise SystemExit("the timed frame is not in parity with the oracle: %s" % line["parity"])
            line["cpu_baseline"] = {"value": rays / sec / 1e6, "unit": "Mrays/s", "cores": threads, "kind": "port",
                                    "sample": sample, "frames_per_s": 1.0 / sec,
                                    "single_thread": {"value": r1 / s1 / 1e6, "unit": "Mrays/s", "cores": 1, "frames_per_s": done1 / (s1 * H),
                                                      "sample": "%d rows (windows of 8 rows spread over the frame), scaled to the frame" % done1},
                                    "note": "C++ restatement of the reference (oracle/), g++ -O2; the D reference cannot be built here"}
        print(json.dumps(line), flush=True)

    if world > 1:
        dist.barrier(group=cpu_group)
        dist.destroy_process_group()
    c2.shutdown()


def executed_fractions(workload, kernel_ms, peaks):
    """What the hardware executed for one frame of `workload` (profiles/executed.json: thread-level FP32 / FP64 FLOPs and
    warp instructions of the render kernel, extracted from a committed ncu report by profiles/ncu_executed.py) against the
    time measured in THIS run: fractions of the measured FP32 / FP64 FMA peaks and of the issue slots."""
    p = os.path.join(ROOT, "profiles", "executed.json")
    ex = (json.load(open(p)) if os.path.exists(p) else {}).get(workload)
    if not ex or not kernel_ms:
        return None
    t = kernel_ms * 1e-3
    slots = peaks["sms"] * 4 * peaks["sm_mhz_effective"] * 1e6 * t   # 4 SMSPs per SM, one warp instruction per clock each
    return {"fp32_flop": ex["fp32_flop"], "fp64_flop": ex["fp64_flop"], "warp_inst": ex["warp_inst"],
            "fp32_frac": ex["fp32_flop"] / t / 1e12 / peaks["fp32_tflops"], "fp64_frac": ex["fp64_flop"] / t / 1e12 / peaks["fp64_tflops"],
            "issue_frac": ex["warp_inst"] / slots, "kernel": ex.get("kernel"), "source": ex.get("source"),
            "note": "counts from the ncu report named in `source` (same kernel build); time and peaks from this run; "
                    "sm clock = the FFMA micro-benchmark's effective clock"}


def C_sizeof_frame_blocks(api):
    import ctypes as C
    return C.sizeof(api.Camera) + C.sizeof(api.Settings)


if __name__ == "__main__":
    main()
