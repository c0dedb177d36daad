"""Gumbel MuZero search (ge_gumbel_root / ge_gumbel_select / ge_gumbel_result, graphenvs_b200.GumbelMCTS) against PUCT
(graphenvs_b200.MCTS): what a simulation round costs, split by launch, and what the decoded episodes return.

For every workload (the shapes of profiles/mcts.py: bench.WORKLOADS, G = the bench's env count / 16 instances, halved until the
tree and its records fit in 16 GB at S = 64), float32 logits and values from a fixed table policy (tab[g % 64, head]):
  round_us        per simulation round at S = 16, every search from the batch's reset state, split by events between the
                  launches of every round: select (ge_gumbel_select / ge_mcts_select), fork_step (ge_state_load + ge_step),
                  policy (the table lookup), save (ge_state_save), expand_backup (ge_mcts_expand); for Gumbel also
                  root_us (ge_gumbel_root, once per search) and result_us (ge_gumbel_result, once per search)
  search_us       one whole search (start + 16 simulations + the readout), device events around it
  decode          mean return and solution cost of run() over the first 256 instances (one search per move), Gumbel at
                  S = 4 / 8 / 16 (max_considered 16) and PUCT at S = 16 / 64, with its wall time
One JSON line per (workload, search, S), with the card name, power limit and max SM clock read in the same run.

    python profiles/gumbel_mcts.py --out profiles/r08_gumbel_mcts.jsonl [--workloads cfg2_longest_path,...]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from beam_search import gpu_identity  # noqa: E402

DEFAULT = "cfg2_longest_path,cfg3_mst,cfg5_multicast,cfg5_distcenter"
S_ROUND = 16
TREE_BYTES = 16e9
TABLES = 64
G_DECODE = 256
DECODE = [("gumbel", 4), ("gumbel", 8), ("gumbel", 16), ("puct", 16), ("puct", 64)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--workloads", default=DEFAULT)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("gumbel_mcts.py measures on a CUDA device; none found")
    import bench
    import graphenvs_b200 as ge
    from graphenvs_b200 import BatchedGraphEnv, _native
    from graphenvs_b200.mcts import _ptr
    from graphenvs_b200.policy import _DTYPES

    ident = gpu_identity()
    dev_name = torch.cuda.get_device_name(0)
    out = open(args.out, "w")

    def emit(line):
        line.update({"gpu": dev_name, "nvidia_smi": ident, "time": time.strftime("%Y-%m-%dT%H:%M:%S")})
        print(json.dumps(line), flush=True)
        out.write(json.dumps(line) + "\n")
        out.flush()

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def timed_search(m, policy, gumbel):
        """One search with events between the launches of every round; per-round means in µs."""
        leaf = m.leaf
        marks = []
        t0 = ev()
        if gumbel:
            m.start(policy, t=0)
        else:
            m.start(policy)
        t1 = ev()
        for k in range(1, m.S + 1):
            a = ev()
            m.tree.flags = (leaf.desc.flags & 16) | m._tree_flags
            m._select(k)
            b = ev()
            leaf.load_states(m.records, m.load_index)
            leaf.step_async(m.sel_action)
            c = ev()
            logits, value = m._policy_out(policy(leaf))
            d = ev()
            leaf.save_states(out=m._node_records[k])
            e = ev()
            _native.check(leaf.lib.ge_mcts_expand(C.byref(m.tree), k, C.byref(leaf.desc), _ptr(leaf.reward), _ptr(logits),
                                                  _DTYPES[logits.dtype], _ptr(value), leaf._stream()))
            f = ev()
            marks.append((a, b, c, d, e, f))
        m.k = m.S
        r0 = ev()
        if gumbel:
            _native.check(leaf.lib.ge_gumbel_result(C.byref(m.tree), C.byref(m.params), _ptr(m._action), _ptr(m._policy),
                                                    _ptr(m._completed_q), leaf._stream()))
        r1 = ev()
        torch.cuda.synchronize()
        res = {name: sum(mk[i].elapsed_time(mk[i + 1]) for mk in marks) * 1e3 / m.S
               for i, name in enumerate(("select", "fork_step", "policy", "save", "expand_backup"))}
        res["start_us"] = t0.elapsed_time(t1) * 1e3
        res["result_us"] = r0.elapsed_time(r1) * 1e3
        return res

    for wl in args.workloads.split(","):
        env_id, N, E, kw, Bb, _, _ = bench.WORKLOADS[wl]
        G0 = Bb // 16
        src = BatchedGraphEnv(env_id, G0, N, E, **dict(kw))
        src.generate(seed=bench.SEED)
        A, AW, R = src.desc.A, src.desc.AW, src.record_bytes()
        per_node = R + 8 * A + 4 * AW + 29
        G = G0
        while G > 32 and per_node * (64 + 1) * G > TREE_BYTES:
            G //= 2
        venv = src.like(G)
        venv.gather_instances(src, torch.arange(G, dtype=torch.int32, device="cuda"))
        venv.reset()
        gen = torch.Generator(device="cuda").manual_seed(5)
        tab = torch.randn((TABLES, N, A), generator=gen, device="cuda")
        vtab = torch.randn((TABLES, N), generator=gen, device="cuda")

        def policy_for(n):
            rows = torch.arange(n, device="cuda") % TABLES

            def policy(env):
                h = env.t["head"].long().clamp(0, N - 1)
                return tab[rows, h], vtab[rows, h]
            return policy

        # ---- round cost at S = 16
        pol = policy_for(G)
        for name in ("gumbel", "puct"):
            m = ge.GumbelMCTS(venv, S_ROUND, seed=1) if name == "gumbel" else ge.MCTS(venv, S_ROUND)
            m.search(pol)                                       # warm-up of every shape
            torch.cuda.synchronize()
            reps, whole = [], []
            for _ in range(args.reps):
                e0 = ev()
                m.search(pol)
                e1 = ev()
                e1.synchronize()
                whole.append(e0.elapsed_time(e1) * 1e3)
                reps.append(timed_search(m, pol, name == "gumbel"))
            med = {k: sorted(r[k] for r in reps)[len(reps) // 2] for k in reps[0]}
            rnd = sum(med[k] for k in ("select", "fork_step", "policy", "save", "expand_backup"))
            emit({"kind": "round", "workload": wl, "env_id": env_id, "search": name, "G": G, "S": S_ROUND, "A": A, "reps": args.reps,
                  "round_us": {k: round(med[k], 2) for k in ("select", "fork_step", "policy", "save", "expand_backup")},
                  "round_us_sum": round(rnd, 2), "start_us": round(med["start_us"], 1),
                  "result_us": round(med["result_us"], 1) if name == "gumbel" else None,
                  "search_us": round(sorted(whole)[len(whole) // 2], 1), "search_us_all": [round(x, 1) for x in whole]})
            del m
        # ---- decode quality over the first G_DECODE instances
        Gd = min(G_DECODE, G)
        dv = venv.like(Gd)
        dv.gather_instances(venv, torch.arange(Gd, dtype=torch.int32, device="cuda"))
        dv.reset()
        pol = policy_for(Gd)
        for name, S in DECODE:
            m = ge.GumbelMCTS(dv, S, seed=1) if name == "gumbel" else ge.MCTS(dv, S)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = m.run(pol)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            f = res.found
            emit({"kind": "decode", "workload": wl, "env_id": env_id, "search": name, "G": Gd, "S": S, "moves": res.steps,
                  "found": int(f.sum()), "mean_return": float(res.ret[f].mean()) if f.any() else None,
                  "mean_solution_cost": float(res.solution_cost[f].mean()) if f.any() else None,
                  "solved": int(res.solved.sum()), "wall_s": round(wall, 2)})
            del m
        del venv, dv, src, tab, vtab
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
