"""Where does an end-to-end host step go?  Wall-clock (perf_counter) of small CUDA graphs replayed on a side stream with a
stream sync, config 2 (LongestPath N=50 E=200 p=2, 65,536 envs): launch+sync floor, each copy alone, the kernel alone,
ge_step_host (single pass) and ge_step_host_pipelined with 1..8 chunks.   python profiles/e2e_breakdown.py [B]"""
import json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from graphenvs_b200 import BatchedGraphEnv

B = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
env = BatchedGraphEnv("LongestPath-v0", B, 50, 200, parenting=2, auto_reset=True)
env.generate(seed=1)
env.reset()
blk, h_rew, h_flg, h_cost, h_bits = env.host_io()
h_act = torch.zeros(B, dtype=torch.int32).pin_memory()
side = torch.cuda.Stream()
torch.cuda.synchronize()


def wall(fn, n=200, warm=20):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    return 1e6 * (time.perf_counter() - t0) / n


def graph_of(body):
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        body()                      # warm-up outside capture
        side.synchronize()
        with torch.cuda.graph(g, stream=side):
            body()

    def run():
        with torch.cuda.stream(side):      # replay() launches on the CURRENT stream
            g.replay()
        side.synchronize()
    return run


out = {"B": B}
tiny = torch.zeros(4, device="cuda")
out["graph_launch_plus_sync_floor_us"] = wall(graph_of(lambda: tiny.add_(1)))
d_act = env.actions_dev
out["h2d_actions_us"] = wall(graph_of(lambda: d_act.copy_(h_act, non_blocking=True)))
io_dev = env._io
out["d2h_results_one_copy_us"] = wall(graph_of(lambda: blk.copy_(io_dev, non_blocking=True)))
out["d2h_bytes"] = int(io_dev.numel())
env.sample_actions(3, 0)
out["kernel_only_us"] = wall(graph_of(lambda: env.step_sampled(3, 0)))
for name, kw in [("single", dict(pipelined=False)), ("pipelined_1", dict(pipelined=True, chunks=1)), ("pipelined_2", dict(pipelined=True, chunks=2)),
                 ("pipelined_3", dict(pipelined=True, chunks=3)), ("pipelined_4", dict(pipelined=True, chunks=4))]:
    stepper = env.host_stepper(h_act, h_rew, h_flg, h_cost, None, h_bits, stream=side, **kw)

    def one():
        env.sample_actions(3, 1)
        h_act.copy_(env.actions_dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        stepper()
        return time.perf_counter() - t0
    for _ in range(10):
        one()
    ts = [one() for _ in range(100)]
    out["ge_step_host_%s_us" % name] = 1e6 * float(np.mean(ts))
    out["ge_step_host_%s_us_min" % name] = 1e6 * float(np.min(ts))
print(json.dumps(out))
