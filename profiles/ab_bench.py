#!/usr/bin/env python
"""A/B timing of library builds on the same GPU, alternated run by run.

  python profiles/ab_bench.py --lib base=build_variants/base --lib new=chess2rt_b200 --workload c1 --workload c0 --runs 3

For each workload it runs `bench.py --workload W --no-cpu-baseline --no-scaling-target --dump-outputs DIR` once per library
directory (C2RT_LIB_DIR, see chess2rt_b200/api.py) in the order A B A B ..., `--runs` times each.  It prints every run's
ms_per_step (with the e2e and interactive legs' times beside it), the median and spread (max - min) per variant, and whether
the frames the variants dumped are np.array_equal.
A variant directory holds libc2rt.so and libc2rt_host.so (chess2rt_b200/build.py build_variant, or a copy of another build).
Frames and bench outputs go to a temporary directory unless --out is given."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(lib_dir, workload, steps, warmup, dump_dir):
    env = dict(os.environ, C2RT_LIB_DIR=os.path.abspath(os.path.join(ROOT, lib_dir)))
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", workload, "--steps", str(steps),
           "--warmup", str(warmup), "--no-cpu-baseline", "--no-scaling-target", "--dump-outputs", dump_dir]
    p = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True)
    if p.returncode != 0:
        raise SystemExit(f"bench.py failed for {lib_dir} on {workload} (exit {p.returncode}):\n{p.stdout[-2000:]}\n{p.stderr[-4000:]}")
    line = [l for l in p.stdout.splitlines() if l.startswith("{")][-1]
    return json.loads(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", required=True, metavar="NAME=DIR", help="a variant: name and library directory")
    ap.add_argument("--workload", action="append", required=True)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", help="keep the dumped frames and a JSON summary here")
    args = ap.parse_args()
    if args.runs < 3:
        raise SystemExit("--runs: at least 3 runs per variant")
    libs = [tuple(s.split("=", 1)) for s in args.lib]
    if len(libs) < 2 or any(len(v) != 2 for v in libs):
        raise SystemExit("--lib NAME=DIR, at least two of them")
    out = args.out or tempfile.mkdtemp(prefix="c2rt_ab_")
    summary = {}
    for wl in args.workload:
        ms = {name: [] for name, _ in libs}
        legs = {name: {"e2e": [], "interactive": []} for name, _ in libs}
        for r in range(args.runs):
            for name, d in libs:
                res = run_bench(d, wl, args.steps, args.warmup, os.path.join(out, wl, name, str(r)))
                ms[name].append(res["ms_per_step"])
                legs[name]["e2e"].append(res["e2e"]["ms_per_step"])
                legs[name]["interactive"].append(res["interactive"]["ms_per_frame"] if res.get("interactive") else float("nan"))
                print(f"{wl} run {r} {name:>12}: {res['ms_per_step']:.5f} ms/step (e2e {legs[name]['e2e'][-1]:.4f} ms, "
                      f"interactive {legs[name]['interactive'][-1]:.4f} ms)", flush=True)
        frames = {name: [np.load(os.path.join(out, wl, name, str(r), "frame.npy")) for r in range(args.runs)] for name, _ in libs}
        ref = frames[libs[0][0]][0]
        same = {name: all(np.array_equal(f, ref) for f in fs) for name, fs in frames.items()}
        summary[wl] = {}
        for name, _ in libs:
            v = ms[name]
            summary[wl][name] = {"ms_per_step": v, "median": statistics.median(v), "spread": max(v) - min(v),
                                 "e2e_ms": legs[name]["e2e"], "interactive_ms": legs[name]["interactive"],
                                 "frames_equal_to_" + libs[0][0]: same[name]}
            print(f"{wl} {name:>12}: median {statistics.median(v):.5f} ms, spread {max(v) - min(v):.5f} ms "
                  f"(min {min(v):.5f}, max {max(v):.5f}); e2e median {statistics.median(legs[name]['e2e']):.4f} ms, interactive median "
                  f"{statistics.median(legs[name]['interactive']):.4f} ms; frames np.array_equal to {libs[0][0]} run 0: {same[name]}",
                  flush=True)
        base = statistics.median(ms[libs[0][0]])
        for name, _ in libs[1:]:
            print(f"{wl} {name} / {libs[0][0]} median ratio: {statistics.median(ms[name]) / base:.4f}", flush=True)
    with open(os.path.join(out, "ab_summary.json"), "w") as f:
        json.dump(summary, f, indent=1)
    print(json.dumps(summary))
    if not all(s["frames_equal_to_" + libs[0][0]] for wl in summary.values() for s in wl.values()):
        raise SystemExit("frames differ between variants")


if __name__ == "__main__":
    main()
