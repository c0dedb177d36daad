#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched GraphEnvs hot path on N B200s (one rank per GPU).

One bench "step" = one pass of the hot path over one batch: sample one valid action per env from
the current mask (README.md:54-68 loop; device counter RNG) and apply Env.step() + the new
Env._get_mask() to all B resident envs, auto-reset on done.  Workloads are BASELINE.json's
configs; the default is configs[1] (LongestPath-v0 N=50 E=200 parenting=2, 65,536 envs per GPU).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

`--impl reference` times the CPU implementation of the same path (the C restatement of the
reference in oracle/, OpenMP over envs, all host threads) on a bounded sample of the workload.

`--dump-outputs DIR` writes what the last timed step of the headline workload returned to its caller
(step_outputs) as DIR/<name>.npy; instances and actions are seeded, so two builds run with the same
arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# name -> (env_id, n_nodes, n_edges, kwargs, envs per GPU, survey bytes per env-step (SURVEY.md 8d), description)
WORKLOADS = {
    "cfg2_longest_path": ("LongestPath-v0", 50, 200, dict(parenting=2, weighted=True), 65536, 1940,
                          "LongestPath-v0 n_nodes=50 n_edges=200 weighted parenting=2, 65536 envs/GPU"),
    "cfg1_shortest_path": ("ShortestPath-v0", 10, 20, dict(weighted=True), 65536, 100,
                           "ShortestPath-v0 n_nodes=10 n_edges=20 weighted, 65536 envs/GPU"),
    "cfg3_mst": ("SteinerTree-v0", 100, 500, dict(n_dests=99, weighted=True, is_eval_env=True), 32768, 5500,
                 "SteinerTree-v0 (MST, n_dests=99) n_nodes=100 n_edges=500 eval, 32768 envs/GPU"),
    "cfg4_tsp_p1": ("TSP-v0", 200, 19900, dict(parenting=1, weighted=True), 16384, 1900,
                    "TSP-v0 n_nodes=200 complete parenting=1, 16384 envs/GPU"),
    "cfg4_tsp_p2": ("TSP-v0", 200, 19900, dict(parenting=2, weighted=True), 16384, 162000,
                    "TSP-v0 n_nodes=200 complete parenting=2, 16384 envs/GPU"),
    "cfg4_mis": ("MaxIndependentSet-v0", 200, 5970, dict(weighted=True), 16384, 300,
                 "MaxIndependentSet-v0 n_nodes=200 n_edges=5970, 16384 envs/GPU"),
    "cfg5_multicast": ("MulticastRouting-v0", 500, 4000, dict(n_dests=3, parenting=4), 131072, 77000,
                       "MulticastRouting-v0 n_nodes=500 n_edges=4000 parenting=4, 131072 envs/GPU"),
    "cfg5_distcenter": ("DistributionCenter-v0", 500, 4000, dict(parenting=2, target_count=100, max_distance=1), 131072,
                        75000, "DistributionCenter-v0 n_nodes=500 n_edges=4000 parenting=2, 131072 envs/GPU"),
    "densest": ("DensestSubgraph-v0", 500, 4000, dict(parenting=1), 65536, 2000,
                "DensestSubgraph-v0 n_nodes=500 n_edges=4000 parenting=1, 65536 envs/GPU"),
    # the reference's ninth id (SURVEY 8 f4; not one of BASELINE's configs): row(head) + one edge weight per step
    "perishable": ("PerishableProductDelivery-v0", 50, 200, dict(n_products=3, parenting=1), 65536, 150,
                   "PerishableProductDelivery-v0 n_nodes=50 n_edges=200 n_products=3 parenting=1, 65536 envs/GPU"),
}
DEFAULT_WORKLOAD = "cfg2_longest_path"
METRIC, UNIT = "env-steps/sec", "env-steps/s"
SEED = 20260101


def layout_bytes_per_step(env):
    """Compulsory HBM bytes per env-step of THIS engine's data layout and algorithm (DESIGN.md section 4):
    state read+write, action in (or the packed mask the in-kernel sampler scans), reward/flags/cost out,
    mask delta or mask rewrite, statistics r/w, plus the graph bytes the env's rule has to read once.
    Useful bytes, not 32-byte sectors: scattered accesses cost more on the wire (see roofline.traffic)."""
    d, N, M = env.desc, env.N, env.M
    nw4 = d.NW * 4
    has_bytes = env.t.get("mask_bytes") is not None
    fixed = 4 + 4 + 4 + 8 + 2 * (4 + 8 + 1) + 2 * 8 + 2 * 8 + 8   # action, reward, flags, sol, head/cost/done rw, acc[2] rw, traj rw, clock
    deg = M / max(N, 1)
    k = env.env_id
    incremental = not (d.flags & 8) and (k in ("SteinerTree-v0",) or (k == "MulticastRouting-v0" and d.parenting >= 2)
                                         or (k == "MaxIndependentSet-v0" and N > 64))
    if incremental:
        has_bytes = False                                  # round 2: the incremental kernels keep only the packed mask current
        sample = d.AW * 4                                  # the sampler walks the packed mask ...
        if env.t.get("mask_cnt") is not None:              # ... or finds the chunk from 16 counts and reads that chunk (+ count updates)
            sample = 32 + ((d.AW + 15) // 16) * 4 + 64
        if k == "MaxIndependentSet-v0":
            return float(fixed + sample + 2 * 8 + 4 + 32 + (1 if has_bytes else 0))
        upd = 2 * deg * (8 + (1 if has_bytes else 0))      # ~deg bits set + ~deg bits cleared (word r/w + byte)
        graph = 8 + 8 + deg * 8                            # col[a], w[a]; rp[v], rp[v+1]; row(v): col + rev / w
        state = nw4 + 8 + 4 + 32                           # tree bits read, one word r/w, target word, counters r/w
        if k == "MulticastRouting-v0":
            graph += 8 + 4 + 8 + 4                         # best[v] (the joining node's distance), dist[v] write, edge bit r/w, max_distance
            if d.parenting >= 3:
                graph += deg * (8 + 4)                     # best[x] read (+ write for about half of them)
        return float(fixed + sample + upd + graph + state)
    mask = d.AW * 4 * 2 + (d.AP if has_bytes else 0)       # old mask read, new written, bytes written
    state = 2 * nw4
    if k == "ShortestPath-v0":
        graph = nw4 + 8
    elif k in ("LongestPath-v0", "TSP-v0"):
        if env.desc.parenting < 2:
            rows = 2                                       # N(head) for the weight rank, N(a) for the next mask
        elif N <= 64 or k == "LongestPath-v0":
            rows = N                                       # the search may touch every row of the bit-matrix
        else:
            rows = min(N, 4 + 2 * N / max(deg, 1.0))       # TSP p=2 on N > 64: spanning search + the few internal candidates
        graph = rows * nw4 + (8 if N <= 64 else 16)
    elif k == "SteinerTree-v0":
        graph = 0.5 * (M * 4 + (N + 1) * 4) + 12 + nw4      # rows of tree nodes: on average half of the CSR
    elif k == "MulticastRouting-v0":
        graph = 0.5 * (M * 8 + (N + 1) * 4) + N * 4 + 12 + nw4 + 2 * d.MW * 4
    elif k == "DistributionCenter-v0":
        # cutoff SSSP ball: with cutoff c and smallest weight w only nodes within c - w are expanded; measured ~22 rows
        # at N=500 E=4000 c=1 (DESIGN.md); each row = 2 row_ptr + deg * (col 4 + w64 8); + in-range rows of the
        # still uncovered targets (about half of them on average) + covered/taken/target sets
        # round 2 (csrc/ge_dc.cu): ~27 rows are expanded at N=500 E=4000 c=1, and of a weight-sorted row only the prefix that
        # can stay within the cutoff is read (~45 % of it), 4 bytes per edge (col | code)
        rows = 27 if (N == 500 and M == 8000) else max(1.0, min(N, 1 + deg + deg * deg * 0.06))
        # (with ge_batch.dc_rows the rows sit at a fixed stride: no row_ptr pair per expanded row)
        graph = rows * ((0 if env.t.get("dc_rows") is not None else 8) + 0.45 * deg * 4) + 0.5 * d.n_targets * (nw4 + 4) + 4 + 4 * nw4
    elif k == "DensestSubgraph-v0":
        graph = nw4 + 16 + 2 * nw4
    elif k == "PerishableProductDelivery-v0":
        graph = nw4 + 8 + deg * 12 + 8 * d.n_dests + 4       # row(head) bits, the head's CSR row scanned for the edge, pickups / dropoffs
        state = 2 * (4 + 16)                                  # head, counters
    else:  # MaxIndependentSet (lane family)
        graph = 4
    return float(fixed + mask + state + graph)


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (ts, r) in self.rows if t0 - 0.05 <= ts <= t1 + 0.15] or [r for _, r in self.rows]
        sm, mx, reasons, pw = [], [], set(), []
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": float(max(pw))}


DUMP_BYTES = 63_000_000      # array bytes of --dump-outputs: with the .npy headers the files stay under 64 MB


def step_outputs(env, budget=DUMP_BYTES):
    """What a caller of the timed step (ge_step_sampled) receives for every env, as float arrays: the action drawn, reward,
    the four flag fields, solution_cost and the packed valid-action mask expanded to [envs, A].  A batch whose arrays would
    exceed `budget` bytes is cut to a fixed, seeded sample of envs; env_index says which."""
    import torch
    B, A = env.B, env.desc.A
    per_env = 8 + 8 + 4 + 4 * 4 + 8 + 4 * A
    idx = np.arange(B)
    if B * per_env > budget:
        idx = np.sort(np.random.default_rng(0).choice(B, budget // per_env, replace=False))
    ti = torch.as_tensor(idx, device=env.reward.device)
    flags = env.flags[ti].cpu().numpy()
    bits = env.t["mask_bits"][ti].cpu().numpy()
    mask = np.unpackbits(bits.view(np.uint8), axis=1, bitorder="little")[:, :A]
    return {"env_index": idx.astype(np.float64), "action": env.actions_dev[ti].cpu().numpy().astype(np.float64),
            "reward": env.reward[ti].cpu().numpy().astype(np.float32), "done": flags[:, 0].astype(np.float32),
            "solved": flags[:, 1].view(np.int8).astype(np.float32), "status": flags[:, 2].astype(np.float32),
            "has_mask": flags[:, 3].astype(np.float32), "solution_cost": env.solution_cost[ti].cpu().numpy().astype(np.float64),
            "mask": mask.astype(np.float32)}


def host_policy(rng, mask):
    """Uniform valid action per env from a bool[B, A] mask (the README loop's np.random.choice)."""
    r = rng.random(mask.shape, dtype=np.float32)
    r[~mask] = -1.0
    return r.argmax(axis=1).astype(np.int32)


# ------------------------------------------------------------------ CPU side (oracle port of the reference)
def cpu_sample_envs(wl, n_envs, seed=1000):
    """Host-generated instances (the reference's own draws, graphenvs_b200/instances.py) wrapped in oracle envs."""
    import random

    import cuda_util as cu
    from graphenvs_b200.instances import generate_instance
    from graphenvs_b200.spec import check_ctor_args
    from oracle import oracle as orc
    env_id, N, E, kw, _, _, _ = WORKLOADS[wl]
    p = check_ctor_args(env_id, N, E, dict(kw))
    envs = []
    for b in range(n_envs):
        random.seed(seed + b)
        np.random.seed(seed + b)
        ins = generate_instance(env_id, p)
        if env_id == "MulticastRouting-v0":  # multicast_routing.py:98-103 with the oracle's own fp64 SSSP
            tmp = cu.oracle_from_instance(env_id, ins, p)
            dist = tmp.sssp(0)
            ft = max(dist[t] for t in ins.dests)
            ins.max_distance = float(np.float32(ins.u01 * (dist.max() - ft) + ft))
        envs.append(cu.oracle_from_instance(env_id, ins, p))
    return envs, orc


def cpu_rate(wl, budget_s, n_envs=None):
    """env-steps/s of the oracle port with all host threads; each pass = one env-step over the sample."""
    env_id, N, E, kw, B, _, _ = WORKLOADS[wl]
    if n_envs is None:
        n_envs = int(min(B, max(64, 4_000_000 // (N * N + 2 * E))))
    t_gen = time.time()
    envs, orc = cpu_sample_envs(wl, n_envs)
    t_gen = time.time() - t_gen
    cores = orc.set_threads(0)        # all host threads (torchrun exports OMP_NUM_THREADS=1)
    orc.rollout(envs, 2, SEED, t0=0)  # warm-up (page in, spawn the OpenMP team)
    t, steps = 2, 0
    t0 = time.perf_counter()
    while True:
        orc.rollout(envs, 1, SEED, t0=t)
        t += 1
        steps += 1
        if time.perf_counter() - t0 >= budget_s:
            break
    dt = time.perf_counter() - t0
    return {"value": n_envs * steps / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d host-generated envs x %d passes (%.1f s; instance generation %.1f s untimed), oracle/graphenvs_oracle.c "
                      "OpenMP over envs" % (n_envs, steps, dt, t_gen)}


def run_reference(args):
    """--impl reference: rank 0 times the CPU port; other ranks exit."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    wl = args.workload
    env_id, N, E, kw, B, _, desc = WORKLOADS[wl]
    n_envs = int(min(B, max(64, 4_000_000 // (N * N + 2 * E))))
    envs, orc = cpu_sample_envs(wl, n_envs)
    cores = orc.set_threads(0)        # all host threads (torchrun exports OMP_NUM_THREADS=1)
    t = 0
    for _ in range(max(args.warmup, 1)):
        orc.rollout(envs, 1, SEED, t0=t)
        t += 1
    t0 = time.perf_counter()
    for _ in range(args.steps):
        orc.rollout(envs, 1, SEED, t0=t)
        t += 1
    dt = time.perf_counter() - t0
    val = n_envs * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64/f32 + bitsets", "data": "synthetic",
            "config": {"workload": desc, "name": wl, "envs_per_step": n_envs,
                       "note": "CPU port of the reference path (pure-Python reference cannot travel to the GPU box); "
                               "each step = one env-step over a bounded sample of the workload"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d host-generated envs x %d passes, OpenMP over envs" % (n_envs, args.steps)},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------ GPU side
CFG5_TOTAL_ENVS = 524288          # per env kind: 524,288 Multicast + 524,288 DistributionCenter = BASELINE configs[4]'s 1M envs
_PY_REF = os.path.join(ROOT, "profiles", "r02_python_reference_cpu.json")


def python_reference_entry(wl):
    """The unmodified reference's own gymnasium loop (pure Python + networkx) for this workload, as RECORDED on the build
    container by oracle/time_python_reference.py (it cannot run on the GPU box: no networkx, no /root/reference)."""
    try:
        j = json.load(open(_PY_REF))
        c = j["configs"][wl]
        return {"one_core_step_only_steps_per_s": c["one_core"]["step_only_steps_per_s"],
                "one_core_incl_reset_steps_per_s": c["one_core"]["incl_reset_steps_per_s"],
                "all_cores_steps_per_s": c["all_cores"]["step_only_steps_per_s"], "cores": c["all_cores"]["processes"],
                "recorded": j["when"], "host": j["host"], "note": c.get("note"),
                "source": "profiles/r02_python_reference_cpu.json (oracle/time_python_reference.py); a stated, dated figure, "
                          "not measured in this run"}
    except Exception:
        return None


class Dist:
    """torch.distributed plumbing of the bench: barrier + MAX / SUM over ranks, no-ops at world 1."""

    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            import torch.distributed as dist
            self.dist = dist
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, vals, op="max"):
        t = self.torch.tensor([float(v) for v in vals], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return [float(x) for x in t]

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


class L2Flush:
    """Between timed steps: a 256 MiB write (evicts the working set; > 126 MB L2) followed by a 256 MiB read (evicts the
    DIRTY flush lines, so the timed kernel does not pay for their write-back).  Per-step CUDA events exclude it."""

    def __init__(self, torch, dev, mode):
        self.torch = torch
        self.buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        self.rd = torch.empty(256 << 20, dtype=torch.uint8, device=dev).view(torch.int64) if mode == "write+read" else None
        self.sink = torch.zeros((), dtype=torch.int64, device=dev)

    def __call__(self):
        self.buf.fill_(1)
        if self.rd is not None:
            self.torch.sum(self.rd, dim=(0,), out=self.sink)


L2_BYTES = 126e6
# sub-batch chains per step in the streaming protocol (graphenvs_b200.batch.SliceStreams); measured sweet spots
STREAM_CHUNKS = {"cfg2_longest_path": 8, "cfg1_shortest_path": 8, "perishable": 4, "cfg3_mst": 2, "densest": 2,
                 "cfg5_multicast": 2, "cfg5_distcenter": 2}   # (profiles/r02_stream_sweep.jsonl)


def measure_streaming(D, flush, wl, B, K, W, env, env0, args, per_launch_bytes, dump=False):
    """Streaming protocol: EXACTLY K steps inside ONE timed region (one CUDA event pair, barrier + synchronize on both sides),
    no flush kernels in it.  The steps rotate over R independent resident batches of B envs whose per-step traffic adds up to
    > 3x L2 (inputs larger than L2: every step finds its batch cold); a workload whose single batch already moves more than
    that per step uses R = 1.  One step of a batch = C sub-batch launches on C free-running stream chains (envs are
    independent: step t+1 of an env only has to follow step t of the same env), launched with GE_FLAG_PDL.
    Returns None when the R batches do not fit in memory (then only the isolated protocol is reported).
    dump: also return step_outputs() of the batch that took the last timed step."""
    import torch
    from graphenvs_b200 import BatchedGraphEnv
    from graphenvs_b200.batch import SliceStreams
    env_id, N, E, kw, _, _, _ = WORKLOADS[wl]
    dev = D.dev
    R = int(max(1, -(-3 * L2_BYTES // max(per_launch_bytes, 1.0))))
    free, _total = torch.cuda.mem_get_info(dev)
    if R > 1 and (R > 48 or (R - 1) * env.memory_bytes() * 1.3 > 0.8 * free):
        return None
    C_ = args.stream_chunks or STREAM_CHUNKS.get(wl, 1)
    envs = [env]
    for r in range(1, R):
        e = BatchedGraphEnv(env_id, B, N, E, device=dev, auto_reset=True, env_id0=env0 + r * B * D.world, **kw)
        e.generate(seed=SEED)
        e.release_w64()
        e.reset()
        e.enable_env_clock()
        envs.append(e)
    for e in envs:
        e.enable_pdl(not args.no_pdl)
    streams, sl = None, None
    if C_ > 1:
        streams = [torch.cuda.Stream(device=dev) for _ in range(C_)]
        sl = [SliceStreams(e, C_, streams=streams) for e in envs]
    for _ in range(max(W, 3)):
        for e in envs:
            e.step_sampled(SEED, 0)
    torch.cuda.synchronize()
    G = max(g for g in range(1, min(K, 1024) + 1) if K % g == 0)
    if G < min(K, 64):     # K without a useful divisor (a prime, say): a graph of up to 1000 steps + one graph for the remainder
        G = min(K, 1000)
    q, r = divmod(K, G)

    def capture(n, first):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            if sl:
                sl[0].fork()
            for i in range(first, first + n):
                if sl:
                    sl[i % R].step_sampled(SEED, 0)
                else:
                    envs[i % R].step_sampled(SEED, 0)
            if sl:
                sl[0].join()
        return g

    graph = capture(G, 0)
    tail = capture(r, q * G) if r else None
    graph.replay()   # untimed (graph upload)
    if tail is not None:
        tail.replay()
    D.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    flush()          # untimed, BEFORE the first event: the first steps start cold too, and while the GPU is busy with it the host
    a.record()       # enqueues the graph behind the event, so the timed region does not begin with the host's launch latency
    for _ in range(q):
        graph.replay()
    if tail is not None:
        tail.replay()
    b.record()
    D.barrier()
    w1 = time.time()
    ms = a.elapsed_time(b)
    total_ms_max = D.reduce([ms], "max")[0]
    outputs = step_outputs(envs[(K - 1) % R]) if dump else None
    for e in envs:
        e.enable_pdl(False)
    n_launch = K * (len(sl[0].bounds) if sl else 1)
    del graph, tail, sl, envs
    torch.cuda.empty_cache()
    return {"total_ms": total_ms_max, "ms_per_step": total_ms_max / K, "steps": K, "replicas": R, "chunks": C_, "pdl": not args.no_pdl,
            "gpu_launches": n_launch, "wall": (w0, w1), "rotation_bytes": per_launch_bytes * R, "outputs": outputs,
            "launch": "CUDA graph of %d steps replayed %d times%s, ONE event pair around all %d steps; step i runs on batch i %% %d; "
                      "each step = %d sub-batch launch(es) on %d stream chain(s)%s" % (G, q, (" + one graph of %d steps" % r) if r else "", K, R, C_, C_, ", programmatic dependent launch" if not args.no_pdl else "")}


def measure_workload(D, flush, wl, B, K, W, args, host_side_policy, envs_total_note=None, sampler=None, seed_env0=None, dump=False):
    """One workload on this rank's B envs: device-timed env-steps/s (value), the end-to-end C-ABI number (e2e), the
    roofline of the step kernel, reset-time costs.  Every rank calls it with the same arguments (barriers inside).
    dump: the result also carries "outputs", step_outputs() of the last timed step of the protocol that gives `value`."""
    import torch
    from graphenvs_b200 import BatchedGraphEnv
    env_id, N, E, kw, _, survey_bytes, desc = WORKLOADS[wl]
    dev, rank, world = D.dev, D.rank, D.world
    env0 = rank * B if seed_env0 is None else seed_env0
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    t_build = time.time()
    env = BatchedGraphEnv(env_id, B, N, E, device=dev, auto_reset=True, env_id0=env0, **kw)
    g0, g1, g2 = ev(), ev(), ev()
    g0.record()
    env.generate(seed=SEED)                       # device generator: same distribution as the reference's reset()
    g1.record()
    env.release_w64()
    env.reset()
    g2.record()
    torch.cuda.synchronize()
    t_build = time.time() - t_build
    reset_block = {"generate_derive_prepare_us_per_env": 1e3 * g0.elapsed_time(g1) / B, "state_reset_us_per_env": 1e3 * g1.elapsed_time(g2) / B,
                   "host_wall_s": t_build}
    lib_bytes = layout_bytes_per_step(env)
    env.enable_env_clock()      # per-env t for the sampler: captured launches draw fresh actions every replay
    fused = args.mode == "fused"
    kernel_name = env.step_kernel_name(sampled=fused)

    def one_step(evs=None):
        flush()
        if evs:
            evs[0].record()
        if fused:                             # action draw + step in one launch (ge_step_sampled):
            env.step_sampled(SEED, 0)         # the step IS the kernel, no event node in between
        else:
            env.sample_actions(SEED, 0)
            if evs:
                evs[1].record()
            env.step_async(env.actions_dev)
        if evs:
            evs[2].record()

    for _ in range(W):
        one_step()
    torch.cuda.synchronize()
    # The step is launch-bound from Python (one ~10-40 us kernel), so the timed steps are replayed from a
    # CUDA graph of G steps; per-step / per-kernel durations come from external event-record nodes in it.
    G = max(g for g in range(1, min(K, 64) + 1) if K % g == 0)
    launch_mode = "CUDA graph of %d steps replayed %d times, external event nodes around every step" % (G, K // G)
    try:
        events = [[torch.cuda.Event(enable_timing=True, external=True) for _ in range(3)] for _ in range(G)]
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for i in range(G):
                one_step(events[i])
        graph.replay()   # one untimed replay (graph upload)
        torch.cuda.synchronize()
        replay = graph.replay
    except Exception as exc:   # no external event nodes on this stack: plain launches, same events, same rules
        torch.cuda.synchronize()
        events = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(G)]
        launch_mode = "plain launches (graph capture unavailable: %s)" % type(exc).__name__

        def replay():
            for i in range(G):
                one_step(events[i])
    if sampler is not None:
        sampler.start()
        time.sleep(0.25)
    D.barrier()
    w0 = time.time()
    step_ms, kern_ms = [], []
    for _ in range(K // G):
        replay()
        torch.cuda.synchronize()
        step_ms += [e[0].elapsed_time(e[2]) for e in events]
        kern_ms += [e[0 if fused else 1].elapsed_time(e[2]) for e in events]
    D.barrier()
    w1 = time.time()
    outputs = step_outputs(env) if dump else None    # before the streaming protocol steps this batch further
    step_ms, kern_ms = np.array(step_ms), np.array(kern_ms)
    assert step_ms.size == K
    total_ms_max, kern_ms_mean = D.reduce([float(step_ms.sum()), float(kern_ms.mean())], "max")
    envs_all = D.reduce([B], "sum")[0]
    iso_value = envs_all * K / (total_ms_max * 1e-3)
    isolated = {"value": iso_value, "unit": UNIT, "ms_per_step": total_ms_max / K, "steps": K, "kernel_ms": kern_ms_mean, "launch": launch_mode,
                "gpu_launches": (1 if fused else 2) * K, "wall_ms_per_step_incl_flush": 1e3 * (w1 - w0) / K,
                "l2": "256 MiB flush %s before every timed step; per-step CUDA event pairs exclude it" % args.flush}
    graph = replay = None                                      # release the isolated-protocol graph
    traffic, traffic_src = None, None
    try:   # measured DRAM bytes per launch of the step kernel (ncu), when this workload/batch was profiled
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(wl)
        if tr and tr.get("envs") == B:
            traffic = tr["bytes_per_launch"]
            traffic_src = "ncu --set full capture of this kernel at this batch (%s); carried from profiles/traffic.json, not measured in this run" % tr.get("source", "profiles/")
    except Exception:
        tr = None
    per_launch = traffic if traffic else (tr["bytes_per_launch"] * B / tr["envs"] if tr else lib_bytes * B)
    stream = None
    if fused and not args.no_streaming:
        try:
            stream = measure_streaming(D, flush, wl, B, K, W, env, env0, args, per_launch, dump=dump)
        except torch.cuda.OutOfMemoryError:       # the R batches did not fit after all: the isolated protocol stands alone
            stream = None
            torch.cuda.empty_cache()
        if D.reduce([0.0 if stream else 1.0], "max")[0] > 0:   # some rank could not stream: nobody does
            stream = None
    clocks = sampler.stop(w0, stream["wall"][1] if stream else w1) if sampler is not None else None
    if stream:
        value, ms_per_step, kern_ms_mean, launch_mode, n_launches = envs_all * K / (stream["total_ms"] * 1e-3), stream["ms_per_step"], stream["ms_per_step"], stream["launch"], stream["gpu_launches"]
        outputs = stream["outputs"]
    else:
        value, ms_per_step, n_launches = iso_value, total_ms_max / K, isolated["gpu_launches"]

    # ---- what an event pair around an (almost) empty kernel measures in the same kind of graph: the share of every timed step
    #      that is launch + event overhead, not kernel (headline only)
    floor_ms = None
    if sampler is not None:
        try:
            tiny = torch.zeros(32, device=dev)
            fe = [[torch.cuda.Event(enable_timing=True, external=True) for _ in range(2)] for _ in range(32)]
            fg = torch.cuda.CUDAGraph()
            with torch.cuda.graph(fg):
                for i in range(32):
                    flush()
                    fe[i][0].record()
                    tiny.add_(1.0)
                    fe[i][1].record()
            for _ in range(2):
                fg.replay()
            torch.cuda.synchronize()
            floor_ms = float(np.mean([a.elapsed_time(b) for a, b in fe]))
        except Exception:
            floor_ms = None

    # ---- end to end through the C ABI with host buffers; the policy between calls is untimed.  Result format: compact
    #      (ge_step_host_compact: reward f32, ONE flag byte, solution_cost f32, packed mask) or full (ge_step_host_pipelined /
    #      ge_step_host: 4 flag bytes, solution_cost f64)
    d = env.desc
    compact = args.e2e_format == "compact" and args.e2e == "pipelined"
    h_act = torch.zeros(B, dtype=torch.int32).pin_memory()
    rng = np.random.default_rng(SEED + rank)
    Ke = max(3, min(K, args.e2e_steps))
    side = torch.cuda.Stream(device=dev)       # a real stream: the host step replays its copy/step/copy sequence as a graph

    def e2e_loop(use_compact, host_policy_on):
        if use_compact:
            h_rew, h_flg, h_cost, h_bits = env.host_io_compact()
        else:
            _blk, h_rew, h_flg, h_cost, h_bits = env.host_io()
        h_bits.copy_(env.t["mask_bits"])
        torch.cuda.synchronize()
        stepper = env.host_stepper(h_act, h_rew, h_flg, h_cost, None, h_bits, stream=side, pipelined=(args.e2e == "pipelined"),
                                   chunks=(None if args.e2e_chunks < 0 else args.e2e_chunks), compact=use_compact)
        tot = 0.0
        D.barrier()
        for k in range(3 + Ke):
            if host_policy_on:                 # README loop on the host: uniform valid action from the mask that came back
                mask = np.unpackbits(h_bits.numpy().view(np.uint8), axis=1, bitorder="little")[:, :d.A].astype(bool)
                h_act.numpy()[:] = host_policy(rng, mask)
            else:                              # large action spaces (up to 8000 edges x 131072 envs): the same draw on the device, copied out
                env.sample_actions(SEED, 7)
                h_act.copy_(env.actions_dev)
            flush()
            torch.cuda.synchronize()
            c0 = time.perf_counter()
            stepper()
            c1 = time.perf_counter()
            if k >= 3:
                tot += c1 - c0
            status = ((h_flg.numpy() >> 3) & 3) if use_compact else h_flg.numpy()[:, 2]
            assert int(status.max()) == 0, "policy produced an invalid action"
        return envs_all * Ke / D.reduce([tot], "max")[0], stepper, (h_rew, h_flg, h_cost, h_bits)

    e2e_val, stepper, (h_rew, h_flg, h_cost, h_bits) = e2e_loop(compact, host_side_policy)
    e2e_chunks = getattr(stepper, "chunks", args.e2e_chunks)
    if args.e2e != "pipelined":
        e2e_how = "ge_step_host: H2D copy of the actions, step kernel, one D2H copy of reward / flags / solution_cost / packed mask, stream sync"
    elif e2e_chunks > 0:
        e2e_how = ("ge_step_host_compact / ge_step_host_pipelined: %d slices on one CUDA graph; the step kernels read the int32 actions straight from the "
                   "pinned host buffer over PCIe (no staging copy), a write-back kernel streams each slice's reward / flags / solution_cost / packed "
                   "mask into the pinned host arrays while the next slice steps; completion polled" % e2e_chunks)
    else:
        e2e_how = ("ge_step_host_compact / ge_step_host_pipelined with chunks = 0: ONE step kernel (actions read from the pinned host buffer) that signals "
                   "per-1024-env progress counters + a concurrent write-back kernel that ships every chunk as soon as it is complete; completion polled")
    e2e_dev_val = e2e_full_val = None
    if host_side_policy:       # the same call with the actions drawn by the device sampler between calls (untimed): the GPU
        e2e_dev_val = e2e_loop(compact, False)[0]   # does not idle for the milliseconds the numpy policy takes (~10 us per call by itself)
        if compact:            # and in the full result format (16 instead of 9 bytes per env next to the mask)
            e2e_full_val = e2e_loop(False, True)[0]
    h2d = B * 4
    d2h = B * (9 if compact else 16) + B * d.AW * 4

    # ---- end to end INCLUDING the observation update for a device-resident consumer: the same host step followed by
    #      ge_obs_graph of the whole batch's node columns (utils.py:14-23: x [B, N, F]); edge tensors are static / reset-time.
    e2e_obs = None
    if args.e2e_obs and hasattr(env, "obs_nodes"):
        xbuf = torch.empty((B, N, env.F), dtype=torch.float32, device=dev)
        fused_obs = args.e2e == "pipelined"
        if fused_obs:     # ge_batch.obs_x: every slice's node columns are rewritten on the write-back lane of the SAME call
            stepper = env.host_stepper(h_act, h_rew, h_flg, h_cost, None, h_bits, stream=side, pipelined=True,
                                       chunks=(None if args.e2e_chunks < 0 else args.e2e_chunks), obs_x=xbuf, compact=compact)
        t_obs = 0.0
        Ko = max(3, min(Ke, 20))
        for k in range(2 + Ko):
            env.sample_actions(SEED, 9)
            h_act.copy_(env.actions_dev)
            flush()
            torch.cuda.synchronize()
            c0 = time.perf_counter()
            stepper()
            if not fused_obs:
                env.obs_nodes(out=xbuf)
                torch.cuda.synchronize()
            c1 = time.perf_counter()
            if k >= 2:
                t_obs += c1 - c0
        t_obs_max = D.reduce([t_obs], "max")[0]
        if fused_obs:     # the rewritten columns are those of the state after the step
            ref_x = env.obs_nodes()
            assert torch.equal(ref_x, xbuf), "obs_x written by the pipelined step differs from ge_obs_nodes"
            env.desc.obs_x = None
        e2e_obs = {"value": envs_all * Ko / t_obs_max, "unit": UNIT, "steps": Ko, "obs_bytes_written_per_env": N * env.F * 4,
                   "what": ("ge_step_host_pipelined with ge_batch.obs_x set: host actions in, results out, and x float32[B, N, F] (the observation's "
                            "node columns, utils.py:14-23) rewritten on the device slice by slice on the write-back lane of the same call")
                           if fused_obs else "ge_step_host (host actions in, results out) + ge_obs_nodes: x float32[B, N, F] rewritten on the device every step"}

    from graphenvs_b200.sharding import reduce_stats
    stats = reduce_stats(env.stats().clone()).cpu().numpy()
    mem = env.memory_bytes()
    del env, stepper
    torch.cuda.empty_cache()

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = lib_bytes * B / (kern_ms_mean * 1e-3) / 1e9
    res = {
        "name": wl, "workload": desc if envs_total_note is None else envs_total_note,
        "value": value, "unit": UNIT, "ms_per_step": ms_per_step, "steps": K, "envs_per_gpu": B, "envs_total": int(envs_all),
        "protocol": ("streaming: K steps in one timed region rotating over %d resident batches (%.0f MB touched per rotation > L2), no flush" %
                     (stream["replicas"], stream["rotation_bytes"] / 1e6)) if stream else "isolated: L2 flush + one event pair per step",
        "streaming": {k: stream[k] for k in ("replicas", "chunks", "pdl", "rotation_bytes")} if stream else None,
        "isolated": isolated,
        "launch": launch_mode, "clocks": clocks,
        "gpu_launches": n_launches,
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": Ke,
                "policy": "host numpy policy on the returned mask" if host_side_policy else "device sampler + copy to the pinned action buffer (untimed)",
                "value_with_device_policy_between_calls": e2e_dev_val,
                "value_full_result_format": e2e_full_val,
                "chunks": e2e_chunks,
                "result_format": ("compact (ge_step_host_compact): reward f32 + 1 flag byte + solution_cost f32 + packed mask" if compact
                                  else "full: reward f32 + 4 flag bytes + solution_cost f64 + packed mask"),
                "timed": "sum of the host-step calls on pinned host buffers, " + e2e_how + "; policy between calls untimed"},
        "e2e_obs": e2e_obs,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "kernel": kernel_name, "kernel_ms": kern_ms_mean,
                     "kernel_ms_what": ("timed region / steps under the streaming protocol (sub-batch launches overlap, so this is the time one "
                                        "full-batch step takes in steady state)" if stream else "mean of the per-step event pairs (isolated protocol)"),
                     "frac_isolated": lib_bytes * B / (isolated["kernel_ms"] * 1e-3) / 1e9 / peak,
                     "event_pair_floor_ms": floor_ms,
                     "event_pair_floor_note": "isolated protocol only: the same event pair around a 32-element add kernel in the same kind of "
                                              "graph = launch + event overhead contained in every isolated kernel_ms (frac_isolated is NOT corrected for it)",
                     "bytes_per_env_step": lib_bytes,
                     "bytes_model": "compulsory bytes of this engine's layout and algorithm per env-step (bench.py:layout_bytes_per_step)",
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s",
                     "survey_bytes_per_env_step": survey_bytes,
                     "frac_if_full_recompute_bytes": survey_bytes * B / (kern_ms_mean * 1e-3) / 1e9 / peak,
                     "frac_if_full_recompute_note": "SURVEY 8(d) bytes of a from-scratch recompute over CSR; NOT this kernel's traffic "
                                                    "(incremental masks / pruned searches move fewer bytes), may exceed 1"},
        "reset": reset_block,
        "episodes": float(stats[0]), "solved": float(stats[1]),
        "memory_gb_per_gpu": mem / 1e9,
    }
    if dump:
        res["outputs"] = outputs
    return res


def compact(res):
    """Entry of the `workloads` array: the figures VERDICT r01 asked the driver-run line to carry per workload."""
    keep = ("name", "workload", "value", "unit", "ms_per_step", "steps", "envs_per_gpu", "protocol", "streaming", "gpu_launches", "e2e", "e2e_obs",
            "reset", "cpu_baseline", "cpu_reference_python", "episodes")
    out = {k: res.get(k) for k in keep if k in res}
    r = res["roofline"]
    out["roofline"] = {k: r[k] for k in ("bound", "achieved", "peak", "unit", "frac", "frac_isolated", "traffic", "kernel", "kernel_ms", "bytes_per_env_step")}
    out["isolated"] = {k: res["isolated"][k] for k in ("value", "ms_per_step", "kernel_ms")}
    out["e2e"] = {k: res["e2e"][k] for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "steps", "policy", "chunks")}
    return out


def feature_costs(D):
    """feature_extraction.generate_features on the device (ge_features) at the configs that produce structural features
    at reset (BASELINE configs[3]) and at config 5's graph size: us per env, CUDA events."""
    import torch
    from graphenvs_b200 import BatchedGraphEnv
    out = {}
    for wl, B in (("cfg4_tsp_p1", 2048), ("cfg4_mis", 2048), ("cfg5_multicast", 2048), ("cfg2_longest_path", 16384)):
        env_id, N, E, kw, _, _, _ = WORKLOADS[wl]
        env = BatchedGraphEnv(env_id, B, N, E, device=D.dev, structural_features=True, **kw)
        env.generate(seed=SEED)       # includes one ge_features pass (warm-up)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        env.compute_features()
        b.record()
        torch.cuda.synchronize()
        out[wl] = {"envs": B, "n_nodes": N, "n_edges": E, "us_per_env": 1e3 * a.elapsed_time(b) / B}
        del env
        torch.cuda.empty_cache()
    return out


def turnover_costs(D, K=300):
    """Reset-INCLUSIVE throughput (VERDICT r01 item 9; every reference reset() builds a new graph, e.g.
    shortest_path.py:47-98): step + instance turnover from a resident pool (graphenvs_b200/pool.py: done envs copy their next
    instance from a bank of prepared instances and are reset; a background stream keeps regenerating banks) next to the
    state-only number under the SAME launch protocol (plain launches from Python, no L2 flush, one event pair around K steps)."""
    import torch
    from graphenvs_b200 import BatchedGraphEnv
    from graphenvs_b200.pool import InstancePool
    out = {}
    for wl in ("cfg1_shortest_path", "cfg5_distcenter"):
        env_id, N, E, kw, B, _, desc = WORKLOADS[wl]
        res = {"workload": desc}
        for mode in ("state_only_auto_reset_same_graph", "pool_turnover"):
            env = BatchedGraphEnv(env_id, B, N, E, device=D.dev, auto_reset=(mode != "pool_turnover"), **kw)
            env.generate(seed=SEED)
            env.reset()
            env.enable_env_clock()
            pool = InstancePool(env, banks=3, seed=11, background=True) if mode == "pool_turnover" else None

            def one():
                env.step_sampled(SEED, 0)
                if pool is not None:
                    pool.turn_over()
            for _ in range(20):
                one()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ep0 = float(env.stats()[0].item())
            a.record()
            for _ in range(K):
                one()
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b) / K
            eps = float(env.stats()[0].item()) - ep0
            r = {"value": B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": K, "episodes_finished": eps,
                 "mean_episode_steps": (B * K / eps) if eps else None, "launches_per_step": 1 if pool is None else 3}
            if pool is not None:
                pool.close()
                r["pool"] = {"banks": pool.G, "instances_resident": pool.G * B, "banks_regenerated_in_background": pool.regenerated,
                             "fresh_instances_generated": pool.regenerated * B, "instances_consumed": eps,
                             "note": "an instance is reused when episodes end faster than the background stream regenerates banks "
                                     "(fresh_instances_generated / instances_consumed = fraction of episodes on a never-seen graph)"}
            res[mode] = r
            del env, pool
            torch.cuda.empty_cache()
        out[wl] = res
    return out


def pin_rank_to_cores(args):
    """One disjoint block of host cores per rank (N > 1): the ranks' launch / completion-polling threads stop competing for
    the same cores.  nvidia-smi topo on the test boxes lists ONE NUMA node and one affinity range for all eight GPUs, so
    there is no closer choice than an even split of that range."""
    world, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if world <= 1 or args.no_pin or not hasattr(os, "sched_setaffinity"):
        return None
    cores = sorted(os.sched_getaffinity(0))
    k = len(cores) // world
    if k < 1:
        return None
    mine = cores[local * k:(local + 1) * k]
    os.sched_setaffinity(0, mine)
    return "%d-%d" % (mine[0], mine[-1])


def run_ours(args):
    import torch
    pinned = pin_rank_to_cores(args)
    D = Dist()
    rank, world = D.rank, D.world
    wl = args.workload
    env_id, N, E, kw, B, survey_bytes, desc = WORKLOADS[wl]
    if args.envs:
        B = args.envs
    K, W = args.steps, args.warmup
    flush = L2Flush(torch, D.dev, args.flush)
    sampler = ClockSampler(D.local) if rank == 0 else None
    t_all = time.time()
    head = measure_workload(D, flush, wl, B, K, W, args, host_side_policy=not args.e2e_device_policy, sampler=sampler,
                            dump=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:      # rank 0's envs
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in head.pop("outputs").items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if world == 1 and not args.no_cpu:
        head["cpu_baseline"] = cpu_rate(wl, args.cpu_seconds)
    head["cpu_reference_python"] = python_reference_entry(wl)

    # ---- every other workload of BASELINE.json (one GPU): same protocol, fewer steps, short CPU sample
    workloads = [compact(head)]
    if world == 1 and not args.only_headline and not args.envs:
        for name in WORKLOADS:
            if name == wl:
                continue
            Kw = min(max(K, 100), CAPS.get(name, 1000))
            r = measure_workload(D, flush, name, WORKLOADS[name][4], Kw, 3, args, host_side_policy=(WORKLOADS[name][1] <= 64))
            if not args.no_cpu:
                r["cpu_baseline"] = cpu_rate(name, args.cpu_seconds_other)
            r["cpu_reference_python"] = python_reference_entry(name)
            workloads.append(compact(r))

    # ---- BASELINE configs[4] as stated: 1M envs in total (524,288 Multicast + 524,288 DistributionCenter) sharded
    #      over the ranks -- STRONG scaling: each rank owns total/world envs of each kind, no data-path collective.
    cfg5 = None
    if not args.only_headline and not args.envs and not args.no_cfg5:
        from graphenvs_b200.sharding import rank_slice
        cfg5 = {"scaling": "strong", "envs_total_per_kind": CFG5_TOTAL_ENVS, "n_gpus": world}
        tot_ms = 0.0
        for name in ("cfg5_multicast", "cfg5_distcenter"):
            lo, cnt = rank_slice(CFG5_TOTAL_ENVS, rank, world)
            r = measure_workload(D, flush, name, cnt, args.cfg5_steps, 3, args, host_side_policy=False, seed_env0=lo,
                                 envs_total_note="%s, %d envs in total sharded over %d GPU(s)" % (WORKLOADS[name][6].split(",")[0], CFG5_TOTAL_ENVS, world))
            cfg5[name] = compact(r)
            cfg5[name]["memory_gb_per_gpu"] = r["memory_gb_per_gpu"]
            tot_ms += r["ms_per_step"]
        cfg5["combined"] = {"value": 2 * CFG5_TOTAL_ENVS / (tot_ms * 1e-3), "unit": UNIT, "ms_per_step_pair": tot_ms,
                            "what": "one step of all 1,048,576 envs = the Multicast launch + the DistributionCenter launch, back to back"}

    feats = feature_costs(D) if (world == 1 and not args.only_headline and not args.envs) else None
    turn = turnover_costs(D) if (world == 1 and not args.only_headline and not args.envs and not args.no_turnover) else None

    if rank == 0:
        line = {
            "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64/f32 + bitsets", "data": "synthetic",
            "config": {"workload": desc, "name": wl, "envs_per_gpu": B, "envs_total": B * world,
                       "instances": "device generator ge_generate (connected G(n,m), reference weight law), seed %d" % SEED,
                       "policy": "uniform valid action, device counter RNG, inside the timed step (%s)" %
                                 ("drawn in the step kernel, ge_step_sampled" if args.mode == "fused" else "ge_sample_actions + ge_step"),
                       "auto_reset": True,
                       "l2": ("inputs larger than L2: the timed steps rotate over %d independent resident batches of %d envs (%.0f MB touched per "
                              "rotation vs 126 MB of L2), no flush inside the timed region" % (head["streaming"]["replicas"], B, head["streaming"]["rotation_bytes"] / 1e6))
                             if head["streaming"] else "256 MiB flush %s between timed steps (per-step CUDA events exclude it)" % args.flush,
                       "launch": head["launch"], "byte_mask": True},
            "clocks": head["clocks"],
            "gpu_launches": head["gpu_launches"],
            "e2e": head["e2e"], "e2e_obs": head["e2e_obs"],
            "roofline": head["roofline"],
            "reset": head["reset"],
            "protocol": head["protocol"], "streaming": head["streaming"], "isolated": head["isolated"],
            "episodes": head["episodes"], "solved": head["solved"], "memory_gb_per_gpu": head["memory_gb_per_gpu"],
            "cpu_reference_python": head["cpu_reference_python"],
            "workloads": workloads,
            "cfg5_strong_scaling": cfg5,
            "feature_extraction_us_per_env": feats,
            "instance_turnover": turn,
            "host_cores_of_rank0": pinned,
            "bench_wall_s": time.time() - t_all,
        }
        if "cpu_baseline" in head:
            line["cpu_baseline"] = head["cpu_baseline"]
        print(json.dumps(line))
    D.close()


# per-workload cap on timed steps in the all-workloads pass (keeps the default run within minutes)
CAPS = {"cfg5_distcenter": 200, "cfg5_multicast": 400, "cfg4_tsp_p2": 400}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0, help="override envs per GPU (headline only)")
    ap.add_argument("--e2e-steps", type=int, default=100)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--cpu-seconds-other", type=float, default=3.0, help="CPU sample per workload in the all-workloads pass")
    ap.add_argument("--cfg5-steps", type=int, default=40)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--only-headline", action="store_true", help="skip the all-workloads pass, config 5 and the feature costs")
    ap.add_argument("--no-cfg5", action="store_true")
    ap.add_argument("--no-turnover", action="store_true")
    ap.add_argument("--no-pin", action="store_true", help="N > 1: do not pin each rank to its own block of host cores")
    ap.add_argument("--no-e2e-obs", dest="e2e_obs", action="store_false")
    ap.add_argument("--flush", default="write+read", choices=["write", "write+read"])
    ap.add_argument("--e2e", default="pipelined", choices=["pipelined", "single"],
                    help="pipelined: ge_step_host in chunks on two streams (copies overlap kernels); single: one copy-in / kernel / copy-out")
    ap.add_argument("--e2e-format", default="compact", choices=["compact", "full"],
                    help="host result format of the end-to-end step: compact = 1 flag byte + float32 solution_cost per env (ge_step_host_compact)")
    ap.add_argument("--e2e-device-policy", action="store_true",
                    help="headline e2e: draw the actions with the device sampler between calls (untimed) instead of the host numpy policy")
    ap.add_argument("--e2e-chunks", type=int, default=-1, help="slices of the pipelined end-to-end step; 0 = streamed write-back (one step kernel + "
                    "concurrent writer fed by progress counters); -1 = auto (streamed for multi-wave batches whose kernel supports it, else 2)")
    ap.add_argument("--no-streaming", action="store_true", help="isolated protocol only (L2 flush + one event pair per step)")
    ap.add_argument("--no-pdl", action="store_true", help="streaming protocol without programmatic dependent launch")
    ap.add_argument("--stream-chunks", type=int, default=0, help="sub-batch chains per step in the streaming protocol (0 = per-workload table)")
    ap.add_argument("--mode", default="fused", choices=["fused", "split"],
                    help="fused: ge_step_sampled (one launch per step); split: ge_sample_actions + ge_step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline workload returned (step_outputs: float32 / float64, "
                         "at most 64 MB, a seeded sample of envs beyond that) as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args)
        return
    if args.gpus > 1 and world == 1:  # convenience: relaunch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29517"] + sys.argv
        sys.exit(subprocess.call(cmd))
    run_ours(args)


if __name__ == "__main__":
    main()
