"""Monte Carlo tree search (ge_mcts_select / ge_mcts_expand, graphenvs_b200.MCTS): what one simulation round costs and where
the time goes, against a torch implementation of the same select and backup and against one policy rollout step.

For every workload (bench.WORKLOADS shapes; G = the bench's env count / 16 instances, halved until the tree and its records
fit in 16 GB), S = 64 simulations, float32 and bfloat16 logits from a fixed table policy (logits = tab[g % 64, head],
value = vtab[g % 64, head]), every search from the batch's reset state:
  search_us       one whole MCTS.search (start + 64 simulations), device events around it
  round_us        per simulation round, split by events between the launches of every round:
                  select, fork_step (ge_state_load + ge_step), policy (the table lookup), save (ge_state_save),
                  expand_backup (ge_mcts_expand)
  torch_search_us the same search with select and expand + backup written in torch (vectorized over instances, one tree
                  level per iteration, a host check per level), the env forks and steps unchanged; its tree is compared
                  with the kernels' (parent, action, N, Wsum bit for bit: trees_agree)
  rollout_step_us sample_logits + step_async over the same G envs: one step of a policy rollout
One JSON line per (workload, dtype), with the card name, power limit and max SM clock read in the same run.

    python profiles/mcts.py --out profiles/r07_mcts.jsonl [--workloads cfg2_longest_path,...]
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
S = 64
TREE_BYTES = 16e9
TABLES = 64


# ------------------------------------------------------------------ the torch implementation of select and expand + backup
def torch_select(m, k):
    """The selection of include/graphenvs_b200.h over all instances at once, one tree level per iteration."""
    import torch
    from graphenvs_b200.mcts import unpack_mask
    G, A, dev = m.G, m.A, m.visits.device
    g = torch.arange(G, device=dev)
    qmin, qmax = m.qmin, m.qmax
    norm = qmax > qmin
    den = torch.where(norm, qmax - qmin, torch.ones_like(qmax))
    s = torch.zeros(G, dtype=torch.long, device=dev)
    depth = torch.zeros(G, dtype=torch.int32, device=dev)
    act = torch.full((G,), -1, dtype=torch.long, device=dev)
    load = torch.full((G,), -1, dtype=torch.long, device=dev)
    active = m.terminal[0] == 0
    while bool(active.any()):
        mask = unpack_mask(m.mask[s, g], A)
        ch = m.child[s, g]
        has = mask & (ch >= 0)
        ci = torch.where(has, ch, 0).long()
        n = torch.where(has, m.visits[ci, g[:, None]], 0)
        Q = m.reward[ci, g[:, None]].double() + m.wsum[ci, g[:, None]] / n.clamp(min=1)
        q = torch.where(has & norm[:, None], (Q - qmin[:, None]) / den[:, None], 0.0)
        sq = torch.sqrt(m.visits[s, g].double())
        u = q + ((m.c_puct * m.prior[s, g].double()) * sq[:, None]) / (1 + n).double()
        u = torch.where(mask, u, float("-inf"))
        ba = u.argmax(dim=1)                                  # the first maximum: ties to the lowest action
        active &= mask.any(dim=1)                             # a dead end is revisited
        bc = ch[g, ba].long()
        depth += active.int()
        exp = active & (bc < 0)
        load = torch.where(exp, s * G + g, load)
        act = torch.where(exp, ba, act)
        active &= ~exp
        s = torch.where(active, bc, s)
        active &= m.terminal[s, g] == 0                       # a terminal child is revisited
    m.sel_node.copy_(s)
    m.sel_action.copy_(act)
    m.load_index.copy_(load)
    m.depth.copy_(depth)


def torch_expand(m, k, logits, value):
    """Expansion and backup of include/graphenvs_b200.h over all instances at once, one tree level per iteration.  The
    priors take lse from ge_masked_log_prob, as the kernel does."""
    import torch
    from graphenvs_b200 import _native
    from graphenvs_b200.policy import _DTYPES
    leaf = m.leaf
    G, A, dev = m.G, m.A, m.visits.device
    g = torch.arange(G, device=dev)
    if k == 0:
        a = torch.full((G,), -1, dtype=torch.long, device=dev)
        par = a.clone()
        create = torch.ones(G, dtype=torch.bool, device=dev)
    else:
        a, par = m.sel_action.long(), m.sel_node.long()
        create = a >= 0
    done = leaf.t["done"] != 0
    mb = leaf.t["mask_bits"]
    lp, ent, lse = (torch.empty(G, device=dev) for _ in range(3))
    zero = torch.zeros(G, dtype=torch.int32, device=dev)
    _native.check(leaf.lib.ge_masked_log_prob(C.c_void_p(logits.data_ptr()), _DTYPES[logits.dtype], G, A, C.c_void_p(mb.data_ptr()),
                                              C.c_void_p(zero.data_ptr()), C.c_void_p(lp.data_ptr()), C.c_void_p(ent.data_ptr()),
                                              C.c_void_p(lse.data_ptr()), leaf._stream()))
    c1 = create[:, None]
    m.prior[k] = torch.where(c1, torch.exp(logits.float() - lse[:, None]), m.prior[k])
    m.child[k] = torch.where(c1, -1, m.child[k])
    m.mask[k] = torch.where(c1, mb, m.mask[k])
    m.parent[k] = torch.where(create, par, -1).int()
    m.action[k] = torch.where(create, a, -1).int()
    m.reward[k] = torch.where(create, leaf.reward if k else torch.zeros_like(leaf.reward), m.reward[k])
    m.terminal[k] = torch.where(create, done.to(torch.uint8), m.terminal[k])
    m.value[k] = torch.where(create, torch.where(done, 0.0, value), m.value[k])
    m.visits[k] = 0
    m.wsum[k] = torch.where(create, 0.0, m.wsum[k])
    if k == 0:
        m.qmin.fill_(float("inf"))
        m.qmax.fill_(float("-inf"))
    else:
        pc = par.clamp(min=0)
        ac = a.clamp(min=0)
        m.child[pc, g, ac] = torch.where(create, k, m.child[pc, g, ac])
    c = torch.where(create, k, par)
    ret = m.value[c, g].double()
    active = torch.ones(G, dtype=torch.bool, device=dev)
    while True:
        n = m.visits[c, g] + active.int()
        w = torch.where(active, m.wsum[c, g] + ret, m.wsum[c, g])
        m.visits[c, g] = n
        m.wsum[c, g] = w
        active &= c != 0
        if not bool(active.any()):
            break
        r = m.reward[c, g].double()
        Q = r + w / n
        m.qmin.copy_(torch.where(active, torch.minimum(m.qmin, Q), m.qmin))
        m.qmax.copy_(torch.where(active, torch.maximum(m.qmax, Q), m.qmax))
        ret = torch.where(active, r + ret, ret)
        c = torch.where(active, m.parent[c, g].long(), c)


def torch_search(m, policy, env):
    """MCTS.search with torch_select / torch_expand in place of the two kernels."""
    leaf = m.leaf
    leaf.gather_instances(env)
    env.save_states(out=m._node_records[0])
    leaf.load_states(m._node_records[0])
    m.sel_action.fill_(-1)
    m.depth.zero_()
    logits, value = m._policy_out(policy(leaf))
    torch_expand(m, 0, logits, value)
    for k in range(1, m.S + 1):
        torch_select(m, k)
        leaf.load_states(m.records, m.load_index)
        leaf.step_async(m.sel_action)
        logits, value = m._policy_out(policy(leaf))
        leaf.save_states(out=m._node_records[k])
        torch_expand(m, k, logits, value)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--workloads", default=DEFAULT)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("mcts.py measures on a CUDA device; none found")
    import bench
    import graphenvs_b200 as ge
    from graphenvs_b200 import BatchedGraphEnv
    from graphenvs_b200 import _native
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

    for wl in args.workloads.split(","):
        env_id, N, E, kw, Bb, _, _ = bench.WORKLOADS[wl]
        G0 = Bb // 16
        src = BatchedGraphEnv(env_id, G0, N, E, **dict(kw))
        src.generate(seed=bench.SEED)
        A, AW, R = src.desc.A, src.desc.AW, src.record_bytes()
        per_node = R + 8 * A + 4 * AW + 29
        G = G0
        while G > 32 and per_node * (S + 1) * G > TREE_BYTES:
            G //= 2
        if G == G0:
            venv = src
        else:
            venv = src.like(G)
            venv.gather_instances(src, torch.arange(G, dtype=torch.int32, device="cuda"))
        del src
        venv.reset()
        m = ge.MCTS(venv, S)
        tm = ge.MCTS(venv, S)
        gen = torch.Generator(device="cuda").manual_seed(5)
        tab32 = torch.randn((TABLES, N, A), generator=gen, device="cuda")
        vtab = torch.randn((TABLES, N), generator=gen, device="cuda")
        rows = torch.arange(G, device="cuda") % TABLES
        for dtype in (torch.float32, torch.bfloat16):
            tab = tab32.to(dtype)

            def policy(env):
                h = env.t["head"].long().clamp(0, N - 1)
                return tab[rows, h], vtab[rows, h]

            m.search(policy)                                   # warm-up of every shape
            torch_search(tm, policy, venv)
            torch.cuda.synchronize()
            agree = all(torch.equal(x, y) for x, y in ((m.parent, tm.parent), (m.action, tm.action), (m.visits, tm.visits),
                                                      (m.wsum.view(torch.int64), tm.wsum.view(torch.int64)),
                                                      (m.qmin, tm.qmin), (m.qmax, tm.qmax)))
            expanded = int((m.visits[1:] > 0).sum())
            depth_max = int(m.depth.max())
            res = {k: [] for k in ("search", "torch_search", "select", "fork_step", "policy", "save", "expand_backup", "rollout_step")}
            for _ in range(args.reps):
                e0 = ev()
                m.search(policy)
                e1 = ev()
                e1.synchronize()
                res["search"].append(e0.elapsed_time(e1) * 1e3)
                e0 = ev()
                torch_search(tm, policy, venv)
                e1 = ev()
                e1.synchronize()
                res["torch_search"].append(e0.elapsed_time(e1) * 1e3)
                # one search again, with events between the launches of every round
                m.start(policy)
                marks = []
                leaf = m.leaf
                for k in range(1, S + 1):
                    t0 = ev()
                    m.tree.flags = leaf.desc.flags & 16
                    _native.check(leaf.lib.ge_mcts_select(C.byref(m.tree), k, leaf._stream()))
                    t1 = ev()
                    leaf.load_states(m.records, m.load_index)
                    leaf.step_async(m.sel_action)
                    t2 = ev()
                    logits, value = m._policy_out(policy(leaf))
                    t3 = ev()
                    leaf.save_states(out=m._node_records[k])
                    t4 = ev()
                    _native.check(leaf.lib.ge_mcts_expand(C.byref(m.tree), k, C.byref(leaf.desc), _ptr(leaf.reward), _ptr(logits),
                                                          _DTYPES[logits.dtype], _ptr(value), leaf._stream()))
                    t5 = ev()
                    marks.append((t0, t1, t2, t3, t4, t5))
                m.k = S
                torch.cuda.synchronize()
                for i, name in enumerate(("select", "fork_step", "policy", "save", "expand_backup")):
                    res[name].append(sum(mk[i].elapsed_time(mk[i + 1]) for mk in marks) * 1e3 / S)
                # one policy rollout step over the same G instances (auto-reset on, as a rollout runs)
                roll = BatchedGraphEnv(env_id, G, N, E, auto_reset=True, **dict(kw))
                roll.generate(seed=bench.SEED)
                roll.reset()
                lg = [tab[rows, roll.t["head"].long().clamp(0, N - 1)].contiguous()]
                roll.sample_logits(lg[0], 1, 0)
                torch.cuda.synchronize()
                n = 50
                e0 = ev()
                for t in range(n):
                    a = roll.sample_logits(lg[0], 1, t)[0]
                    roll.step_async(a)
                e1 = ev()
                e1.synchronize()
                res["rollout_step"].append(e0.elapsed_time(e1) * 1e3 / n)
                del roll
            med = {k: sorted(v)[len(v) // 2] for k, v in res.items()}
            rnd = sum(med[k] for k in ("select", "fork_step", "policy", "save", "expand_backup"))
            emit({
                "workload": wl, "env_id": env_id, "dtype": "bf16" if dtype == torch.bfloat16 else "f32", "G": G, "G_bench_over_16": G0,
                "S": S, "A": A, "AW": AW, "record_bytes": R, "tree_bytes": m.memory_bytes(), "expanded_nodes": expanded,
                "expanded_per_instance": round(expanded / G, 2), "last_depth_max": depth_max, "reps": args.reps,
                "search_us": round(med["search"], 1), "search_us_per_round": round(med["search"] / S, 2),
                "round_us": {k: round(med[k], 2) for k in ("select", "fork_step", "policy", "save", "expand_backup")},
                "round_us_sum_with_events": round(rnd, 2),
                "torch_search_us": round(med["torch_search"], 1),
                "torch_over_kernels": round(med["torch_search"] / med["search"], 2), "trees_agree": agree,
                "rollout_step_us": round(med["rollout_step"], 2),
                "round_over_rollout_step": round(med["search"] / S / med["rollout_step"], 2),
                "us_all": {k: [round(x, 1) for x in v] for k, v in res.items()},
            })
            del tab
        del m, tm, venv, tab32
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
