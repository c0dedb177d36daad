#!/usr/bin/env python
"""One cfg2 batch (LongestPath N=50, E=200, parenting=2, 65,536 envs) stepped back to back on ONE stream with programmatic
dependent launch: every launch becomes resident while the previous one is still writing the state it is about to read, so the
lane step's guessed draw (csrc/ge_lane.cu: the edge weight it prefetches before griddepcontrol.wait) is made from stale state.
This is the worst case of that prefetch; the bench's schedule steps other batches in between.  The batch (40 MB) stays in L2.

  python profiles/lane_pdl_window.py --label change --out profiles/r08_lane_pdl_window.jsonl [--steps K] [--repeats N]
Prints one JSON line per launch mode (PDL, plain) with the card, its power limit and max SM clock, and appends them to --out.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from graphenvs_b200 import BatchedGraphEnv  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--label", required=True, help="build under test, copied into every line")
    ap.add_argument("--out", default=None, help="append the lines to this file")
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    env_id, N, E, kw, B, _, _ = bench.WORKLOADS["cfg2_longest_path"]
    env = BatchedGraphEnv(env_id, B, N, E, device=torch.device("cuda", 0), auto_reset=True, **kw)
    env.generate(seed=bench.SEED)
    env.release_w64()
    env.reset()
    env.enable_env_clock()
    lines = []
    for mode in ("pdl", "plain"):
        env.enable_pdl(mode == "pdl")
        for _ in range(10):
            env.step_sampled(bench.SEED, 0)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(args.steps):
                env.step_sampled(bench.SEED, 0)
        g.replay()
        torch.cuda.synchronize()
        us = []
        for _ in range(args.repeats):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            g.replay()
            b.record()
            torch.cuda.synchronize()
            us.append(a.elapsed_time(b) * 1000.0 / args.steps)
        del g
        us.sort()
        lines.append({"label": args.label, "card": card(), "workload": "cfg2_longest_path", "envs": B, "launch": mode,
                      "schedule": "one batch, one stream, %d steps per CUDA graph" % args.steps, "kernel": env.step_kernel_name(sampled=True),
                      "us_per_step_median": us[len(us) // 2], "us_per_step_min": us[0], "us_per_step_max": us[-1], "repeats": args.repeats})
    for line in lines:
        print(json.dumps(line))
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
