"""Per-env state records and instance replication (csrc/ge_state.cu) against a device copy of the same bytes and against the
torch code a user writes without them.

For every workload (bench.WORKLOADS shapes, generated envs after a few sampled steps), times in us per call:
  save          BatchedGraphEnv.save_states(out=...) of every env
  load          load_states(records, perm), a random permutation of the records
  gather        like(B).gather_instances(env, perm): every static array of a random permutation of the instances
  torch_save    torch.index_select(out=) of every state tensor of env.t (mask_bytes included), one launch per tensor
  torch_load    the same from saved tensors into env.t, gathered by the permutation
  copy_*        a torch copy_ of a buffer moving as many bytes (read + write) as save / load / gather: the copy bandwidth
  step          one step_sampled: what a save + load costs next to a step
Every call is cold in L2 (a 512 MB buffer is zeroed before it, outside its event pair), and the variants alternate within
each repetition.  Bytes per call are counted from the arrays: state sections read and records written for a save, the reverse
(plus the rebuilt byte mask) for a load, and every static array's bytes read and written for a gather.  Writes one JSON line
per workload, with the device name and its power limit.

    python profiles/env_state.py --out profiles/r04_env_state.jsonl [--workloads cfg2_longest_path,...]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DEFAULT = "cfg2_longest_path,cfg3_mst,cfg5_multicast,cfg5_distcenter"
STATE = ("head", "node_bits", "node_bits2", "edge_bits", "dist32", "bestkey", "cost", "counters", "done", "mask_bits", "mask_cnt",
         "acc", "traj")
STATIC = ("row_ptr", "col", "w32", "w64", "adj_bits", "rev", "esrc", "wsort", "wcode", "dc_edges", "dc_rows", "wmin", "wmat",
          "src", "dest", "target_bits", "node_cost", "node_xy", "max_dist32", "targets", "in_range", "heuristic",
          "heuristic_alt", "features", "mask0_bits")


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # the device name from torch is still recorded
        return "nvidia-smi unavailable (%s)" % e


def nbytes(t):
    return t.numel() * t.element_size()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--workloads", default=DEFAULT)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=40)
    ap.add_argument("--warm-steps", type=int, default=6)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("env_state.py measures on a CUDA device; none found")
    import bench
    from graphenvs_b200 import BatchedGraphEnv

    ident = gpu_identity()
    dev_name = torch.cuda.get_device_name(0)
    out = open(args.out, "w")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")

    def timed(fn, n):
        """Median us of n calls, each cold in L2 and between its own pair of events."""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        for i, (s, e) in enumerate(ev):
            flush.zero_()
            s.record()
            fn(i)
            e.record()
        torch.cuda.synchronize()
        t = sorted(s.elapsed_time(e) * 1e3 for s, e in ev)
        return t[n // 2]

    for wl in args.workloads.split(","):
        env_id, N, E, kw, B, _, _ = bench.WORKLOADS[wl]
        env = BatchedGraphEnv(env_id, B, N, E, auto_reset=True, **dict(kw))
        env.generate(seed=bench.SEED)
        env.reset()
        for t in range(args.warm_steps):
            env.step_sampled(1, t)
        torch.cuda.synchronize()
        R = env.record_bytes()
        keys = [k for k in STATE if k in env.t]
        state_bytes = sum(nbytes(env.t[k]) for k in keys) // B
        mask_rebuilt = bool(env.lib.ge_mask_bytes_current(C.byref(env.desc)))
        bytes_save = B * (state_bytes + R)
        bytes_load = B * (R + state_bytes + (env.desc.AP if mask_rebuilt else 0))
        perm = torch.randperm(B, device="cuda").int()
        buf = env.save_states()
        wide = env.like(B)
        wide.gather_instances(env, perm)
        static_keys = [k for k in STATIC if k in wide.t]
        bytes_gather = 2 * sum(nbytes(wide.t[k]) for k in static_keys)
        # the torch path: every state tensor of env.t, the byte mask included (it is what env.mask reads)
        tkeys = keys + (["mask_bytes"] if "mask_bytes" in env.t else [])
        saved = {k: env.t[k].clone() for k in tkeys}
        ar = torch.arange(B, device="cuda")
        perm64 = perm.long()
        copies = {name: (torch.empty(b // 2, dtype=torch.uint8, device="cuda"), torch.empty(b // 2, dtype=torch.uint8, device="cuda"))
                  for name, b in (("save", bytes_save), ("load", bytes_load), ("gather", bytes_gather))}

        def f_save(i):
            env.save_states(out=buf)

        def f_load(i):
            env.load_states(buf, perm)

        def f_gather(i):
            wide.gather_instances(env, perm)

        def f_torch_save(i):
            for k in tkeys:
                torch.index_select(env.t[k], 1 if k == "acc" else 0, ar, out=saved[k])

        def f_torch_load(i):
            for k in tkeys:
                torch.index_select(saved[k], 1 if k == "acc" else 0, perm64, out=env.t[k])

        def copier(name):
            dst, src = copies[name]
            return lambda i: dst.copy_(src)

        def f_step(i):
            env.step_sampled(2, 100 + i)

        step_us = [timed(f_step, args.calls) for _ in range(2)][-1]   # before any load: the envs hold their own states
        variants = [("save", f_save), ("torch_save", f_torch_save), ("copy_save", copier("save")), ("load", f_load),
                    ("torch_load", f_torch_load), ("copy_load", copier("load")), ("gather", f_gather), ("copy_gather", copier("gather"))]
        for _, f in variants:   # warm-up of every shape the timed calls use
            timed(f, 2)
        res = {k: [] for k, _ in variants}
        for r in range(args.reps):
            for k, f in variants:
                res[k].append(timed(f, args.calls))
        med = {k: sorted(v)[len(v) // 2] for k, v in res.items()}
        gbps = lambda b, us: round(b / (us * 1e3), 1)  # noqa: E731
        line = {
            "workload": wl, "env_id": env_id, "B": B, "record_bytes": R, "state_bytes_per_env": state_bytes,
            "mask_bytes_rebuilt_on_load": mask_rebuilt, "static_bytes_per_env": bytes_gather // (2 * B),
            "bytes_per_call": {"save": bytes_save, "load": bytes_load, "gather": bytes_gather},
            "calls_per_window": args.calls, "reps": args.reps,
            "us": {k: round(v, 2) for k, v in med.items()}, "us_all": {k: [round(x, 2) for x in v] for k, v in res.items()},
            "step_sampled_us": round(step_us, 2),
            "GBps": {k: gbps(b, med[k]) for k, b in (("save", bytes_save), ("load", bytes_load), ("gather", bytes_gather))},
            "copy_GBps": {k: gbps(b, med["copy_" + k]) for k, b in (("save", bytes_save), ("load", bytes_load), ("gather", bytes_gather))},
            "frac_of_copy": {k: round(med["copy_" + k] / med[k], 3) for k in ("save", "load", "gather")},
            "torch_launches": {"save": len(tkeys), "load": len(tkeys)}, "launches": {"save": 1, "load": 1, "gather": 1},
            "speedup_vs_torch": {k: round(med["torch_" + k] / med[k], 2) for k in ("save", "load")},
            "save_plus_load_over_step": round((med["save"] + med["load"]) / step_us, 2),
            "gpu": dev_name, "nvidia_smi": ident, "time": time.strftime("%Y-%m-%dT%H:%M:%S"),
        }
        print(json.dumps(line), flush=True)
        out.write(json.dumps(line) + "\n")
        out.flush()
        del env, wide, buf, saved, copies
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
