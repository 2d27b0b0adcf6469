"""Tuning aid: render_solo_kernel's strip width (tiles per CTA, render_kernel.cu solo_strip) swept in one process.

  C2RT_LIB_DIR=build_variants/mb6 python profiles/strip_sweep.py --workload c1 --workload c0 --rounds 5

For each workload it times c2rt_render_device on the full frame with S = 0 (the width the launch picks) and S = 1..8 forced
(C2RT_SOLO_STRIP, read at every launch), the widths alternated round by round: per width and round `--warmup` frames, then
`--steps` frames, each behind a 256 MB fill that flushes the L2, timed with CUDA events around the render; ms per frame = mean.
It prints every round's time, the median and spread per width, its ratio to S = 0, and whether every frame of the call is
np.array_equal to the first one."""
import argparse
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import chess2rt_b200 as c2  # noqa: E402
from bench import RNG_SEED, WORKLOADS  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", action="append", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--widths", default="0,1,2,3,4,5,6,7,8")
    args = ap.parse_args()
    widths = [int(s) for s in args.widths.split(",")]
    c2.init(1, [0])
    print("lib:", os.environ.get("C2RT_LIB_DIR", "chess2rt_b200"), "| device:", torch.cuda.get_device_name(0), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    for name in args.workload:
        path, W, H, over = WORKLOADS[name]
        assert not over, "strip_sweep.py runs workloads without settings overrides"
        scene = c2.HostScene(os.path.join(ROOT, path))
        scene.set_frame_size(W, H)
        handle = scene.device_scene()
        cam, st = scene.frame_blocks(seed=RNG_SEED)
        frame = torch.empty((H, W, 3), dtype=torch.float32, device="cuda")
        ms = {s: [] for s in widths}
        ref, equal = None, True
        for _ in range(args.rounds):
            for s in widths:
                if s:
                    os.environ["C2RT_SOLO_STRIP"] = str(s)
                else:
                    os.environ.pop("C2RT_SOLO_STRIP", None)
                for _ in range(args.warmup):
                    c2.render_device(handle, cam, st, frame.data_ptr(), None, None, stream)
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
                for e0, e1 in ev:
                    flush.fill_(1)
                    e0.record()
                    c2.render_device(handle, cam, st, frame.data_ptr(), None, None, stream)
                    e1.record()
                torch.cuda.synchronize()
                ms[s].append(sum(e0.elapsed_time(e1) for e0, e1 in ev) / len(ev))
                f = frame.cpu().numpy()
                if ref is None:
                    ref = f
                equal = equal and np.array_equal(f, ref)
        os.environ.pop("C2RT_SOLO_STRIP", None)
        base = statistics.median(ms[widths[0]])
        for s in widths:
            v = ms[s]
            print(f"{name} S={s}: " + " ".join(f"{x:.5f}" for x in v) + f"  median {statistics.median(v):.5f} spread "
                  f"{max(v) - min(v):.5f}  ratio {statistics.median(v) / base:.4f}", flush=True)
        print(f"{name}: every frame np.array_equal to the first: {equal}", flush=True)


if __name__ == "__main__":
    main()
