#!/usr/bin/env python
"""Streaming protocol sweep: K steps in ONE timed region (one event pair), no L2 flush -- the steps rotate over R
independent resident batches whose per-step traffic adds up to more than L2, so every step finds its data cold.  Each
step of a batch is C sub-batch launches on C free-running streams (graphenvs_b200.batch.SliceStreams).

  python profiles/stream_sweep.py --workload cfg2_longest_path --chunks 1,2,4,8 [--replicas R] [--steps K]
Prints one JSON line per (C) setting.  --pdl launches every step with programmatic dependent launch (enable_pdl()).
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from graphenvs_b200 import BatchedGraphEnv  # noqa: E402
from graphenvs_b200.batch import SliceStreams  # noqa: E402

L2_BYTES = 126e6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg2_longest_path")
    ap.add_argument("--chunks", default="1,2,4,8")
    ap.add_argument("--replicas", type=int, default=0)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--envs", type=int, default=0)
    ap.add_argument("--pdl", action="store_true", help="step launches may start under the previous launch's tail (GE_FLAG_PDL)")
    args = ap.parse_args()
    wl = args.workload
    env_id, N, E, kw, B, _, desc = bench.WORKLOADS[wl]
    B = args.envs or B
    dev = torch.device("cuda", 0)
    tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(wl, {})
    per_launch = tr.get("bytes_per_launch", 0) * (B / tr.get("envs", B)) if tr else 0
    R = args.replicas or max(1, min(32, int(-(-3 * L2_BYTES // max(per_launch, 1)))))
    envs = []
    for r in range(R):
        e = BatchedGraphEnv(env_id, B, N, E, device=dev, auto_reset=True, env_id0=r * B, **kw)
        e.generate(seed=bench.SEED)
        e.release_w64()
        e.reset()
        e.enable_env_clock()
        envs.append(e)
    torch.cuda.synchronize()
    if args.pdl:
        for e in envs:
            e.enable_pdl()
    mem = sum(e.memory_bytes() for e in envs)
    lib_bytes = bench.layout_bytes_per_step(envs[0])
    for e in envs:
        for _ in range(3):
            e.step_sampled(bench.SEED, 0)
    torch.cuda.synchronize()
    for C in [int(c) for c in args.chunks.split(",")]:
        streams = None
        if C > 1:
            sl = [SliceStreams(e, C) for e in envs]
            streams = sl[0].streams
            for s in sl[1:]:
                s.streams = streams          # slice c of every batch rides stream c
        m = max(1, min(args.steps, 1024) // R)
        G = R * m
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            if C > 1:
                sl[0].fork()
            for i in range(G):
                if C > 1:
                    sl[i % R].step_sampled(bench.SEED, 0)
                else:
                    envs[i % R].step_sampled(bench.SEED, 0)
            if C > 1:
                sl[0].join()
        reps = max(1, args.steps // G)
        graph.replay()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            graph.replay()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / (reps * G)
        print(json.dumps({"workload": wl, "envs": B, "replicas": R, "rotation_bytes": per_launch * R, "chunks": C, "pdl": args.pdl,
                          "steps": reps * G, "us_per_step": 1e3 * ms, "env_steps_per_s": B / (ms * 1e-3),
                          "frac_hbm": lib_bytes * B / (ms * 1e-3) / 1e9 / 6545.3, "mem_gb": mem / 1e9,
                          "kernel": envs[0].step_kernel_name(sampled=True)}), flush=True)
        del graph


if __name__ == "__main__":
    main()
