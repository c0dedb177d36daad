"""GPU: Monte Carlo tree search (ge_mcts_select / ge_mcts_expand, graphenvs_b200.MCTS).  Every kernel family against an exact
float64 reference search that takes its transitions, masks and terminals from the C oracle; tree invariants and full
coverage on tiny instances; whole-episode decoding replayed in the oracle; S = 1 and done roots; CUDA-graph and PDL
scheduling."""
import math
import random

import numpy as np
import pytest
import torch

import cuda_util as cu
import graphenvs_b200 as ge
from graphenvs_b200 import BatchedGraphEnv
from graphenvs_b200.instances import generate_instance
from graphenvs_b200.mcts import unpack_mask
from test_cuda_beam import TINY
from test_cuda_env_state import FAMILIES, IDS, make_batch

pytestmark = pytest.mark.gpu

C_PUCT = 1.25


# ------------------------------------------------------------------ a policy both sides can compute
def _key(g, depth, action):
    return g * 131 + depth * 17 + (action + 1) * 7


def ref_logits(g, depth, action, A):
    k = _key(g, depth, action)
    a = np.arange(A, dtype=np.int64)
    return (((k * 37 + a * 11 + (k * a) % 23) % 29 - 14) * 0.125).astype(np.float32)


def ref_value(g, depth, action):
    return float(np.float32(((_key(g, depth, action) * 13) % 41 - 20) / 8))


def keyed_policy(m, dtype=torch.float32, zero=False):
    """logits and value hashed from (instance, depth of the leaf, action into the leaf) -- m.depth and m.sel_action."""
    G, A = m.G, m.A
    g = torch.arange(G, device="cuda", dtype=torch.int64)
    a = torch.arange(A, device="cuda", dtype=torch.int64)

    def policy(env):
        assert env is m.leaf
        if zero:
            return torch.zeros((G, A), device="cuda", dtype=dtype), torch.zeros(G, device="cuda")
        k = (g * 131 + m.depth.long() * 17 + (m.sel_action.long() + 1) * 7)[:, None]
        logits = (((k * 37 + a * 11 + (k * a) % 23) % 29 - 14).float() * 0.125).to(dtype)
        value = ((k[:, 0] * 13) % 41 - 20).float() / 8
        return logits, value
    return policy


# ------------------------------------------------------------------ the oracle side
class Replayer:
    """One instance: the oracle's mask, last step outputs and return after an action prefix (replayed from reset, cached)."""

    def __init__(self, oe):
        self.oe, self.cache = oe, {}

    def __call__(self, prefix):
        prefix = tuple(prefix)
        if prefix not in self.cache:
            oe = self.oe
            oe.reset_state()
            m, o, ret = oe.mask(reset_patch=True), None, 0.0
            for a in prefix:
                assert o is None or not o["done"], prefix
                o = oe.step(a)
                assert o["status"] == 0, prefix
                ret += o["reward"]
                if o["has_mask"]:
                    m = o["mask"]
            self.cache[prefix] = (np.asarray(m, dtype=bool), o, ret)
        return self.cache[prefix]


def _close(x, y, tol=1e-5):
    return abs(x - y) <= tol * max(1.0, abs(y))


def tree_of(m, g):
    """The device tree of instance g on the host."""
    T = {k: getattr(m, k)[:, g].cpu().numpy() for k in ("parent", "action", "visits", "wsum", "reward", "value", "terminal")}
    T["mask"] = unpack_mask(m.mask[:, g], m.A).cpu().numpy()
    T["prior"] = m.prior[:, g].cpu().numpy()
    T["child"] = m.child[:, g].cpu().numpy()
    T["created"] = np.flatnonzero(T["visits"] > 0)
    T["prefix"] = {}
    for n in T["created"]:
        p, c = [], int(n)
        while c > 0:
            p.append(int(T["action"][c]))
            c = int(T["parent"][c])
        T["prefix"][int(n)] = tuple(reversed(p))
    return T


def reference_search(S, root_terminal, valid_of, step_of, prior_of, value_of, c_puct=C_PUCT):
    """The search of include/graphenvs_b200.h restated in Python floats (float64, correctly rounded, no FMA).
    valid_of(prefix) -> ascending valid actions; step_of(prefix) -> (r, terminal) of the edge into that prefix;
    prior_of(node, a); value_of(depth, action).  Node k is created in simulation k, as on the device."""
    nodes = {}
    qmm = [math.inf, -math.inf]

    def make(k, parent, action, prefix):
        if prefix:
            r, term = step_of(prefix)
        else:
            r, term = 0.0, root_terminal
        depth = len(prefix)
        nodes[k] = dict(parent=parent, action=action, prefix=prefix, r=r, term=term,
                        v=0.0 if term else value_of(depth, action), N=0, W=0.0, children={})

    def backup(n):
        ret = nodes[n]["v"]
        while True:
            nd = nodes[n]
            nd["N"] += 1
            nd["W"] = nd["W"] + ret
            if n == 0:
                break
            Q = nd["r"] + nd["W"] / nd["N"]
            qmm[0], qmm[1] = min(qmm[0], Q), max(qmm[1], Q)
            ret = nd["r"] + ret
            n = nd["parent"]

    make(0, -1, -1, ())
    backup(0)
    for k in range(1, S + 1):
        s, leaf = 0, None
        while not nodes[s]["term"]:
            best, ba, bc = -math.inf, None, None
            sq = math.sqrt(nodes[s]["N"])
            qmin, qmax = qmm
            for a in valid_of(nodes[s]["prefix"]):
                c = nodes[s]["children"].get(a)
                n, q = 0, 0.0
                if c is not None:
                    n = nodes[c]["N"]
                    if qmax > qmin:
                        Q = nodes[c]["r"] + nodes[c]["W"] / n
                        q = (Q - qmin) / (qmax - qmin)
                u = q + ((c_puct * prior_of(s, a)) * sq) / (1 + n)
                if u > best:
                    best, ba, bc = u, a, c
            if ba is None:
                break                                      # a dead end: revisit s
            if bc is None:
                make(k, s, ba, nodes[s]["prefix"] + (ba,))
                nodes[s]["children"][ba] = leaf = k
                break
            s = bc
        backup(s if leaf is None else leaf)
    return nodes, qmm


def check_node_data(m, venv, g, T, rep, dtype):
    """The device's per-node data against the oracle and the policy: terminal flags, rewards, masks and priors."""
    for n in T["created"]:
        p = T["prefix"][n]
        mask, o, _ = rep(p)
        term = bool(o["done"]) if p else bool(venv.t["done"][g].item())
        assert bool(T["terminal"][n]) == term, (g, n)
        if n:
            assert _close(float(T["reward"][n]), o["reward"]), (g, n)
        if term:
            continue
        assert np.array_equal(T["mask"][n], mask), (g, n)
        lg = torch.from_numpy(ref_logits(g, len(p), int(T["action"][n]), m.A)).to(dtype).double()
        lg[~torch.from_numpy(mask)] = -math.inf
        sm = torch.softmax(lg, 0).numpy()
        # float32 rounding of l - lse (|l - lse| < 16: half an ulp is 4.8e-7) and of lse itself
        np.testing.assert_allclose(T["prior"][n][mask], sm[mask], rtol=2e-6, atol=0)


def check_against_reference(m, venv, inst, env_id, dtype=torch.float32, c_puct=C_PUCT):
    res = m.result()
    r_visits, r_q, r_value, r_action = (x.cpu().numpy() for x in (res.visits, res.q, res.value, res.action))
    for g in range(m.G):
        T = tree_of(m, g)
        rep = Replayer(cu.oracle_from_instance(env_id, inst[g], venv.params))
        check_node_data(m, venv, g, T, rep, dtype)
        dev = {p: n for n, p in T["prefix"].items()}
        nodes, qmm = reference_search(
            m.S, bool(venv.t["done"][g].item()),
            valid_of=lambda p: np.flatnonzero(rep(p)[0]).tolist(),
            step_of=lambda p: (float(T["reward"][dev[p]]), bool(rep(p)[1]["done"])),   # the device's float32 rewards
            prior_of=lambda s, a: float(T["prior"][s][a]),                           # the device's priors
            value_of=lambda d, a: ref_value(g, d, a), c_puct=c_puct)
        assert T["created"].tolist() == sorted(nodes), "instance %d: created nodes" % g
        for k, nd in nodes.items():
            tag = "instance %d node %d" % (g, k)
            assert T["prefix"][k] == nd["prefix"] and int(T["parent"][k]) == nd["parent"], tag
            assert int(T["visits"][k]) == nd["N"], tag
            assert float(T["wsum"][k]) == nd["W"], tag          # bit for bit
            assert float(T["value"][k]) == nd["v"], tag
        assert m.qmin[g].item() == qmm[0] and m.qmax[g].item() == qmm[1], g
        # the root outputs
        root = nodes[0]
        for a in range(m.A):
            c = root["children"].get(a)
            assert int(r_visits[g, a]) == (nodes[c]["N"] if c is not None else 0), (g, a)
            q = float(r_q[g, a])
            if c is None:
                assert math.isnan(q)
            else:
                assert q == nodes[c]["r"] + nodes[c]["W"] / nodes[c]["N"], (g, a)
        assert float(r_value[g]) == root["W"] / root["N"]
        vis = [nodes[root["children"][a]]["N"] if a in root["children"] else 0 for a in range(m.A)]
        exp_a = -1 if root["term"] or not root["children"] else int(np.argmax(vis))
        assert int(r_action[g]) == exp_a, g


# ------------------------------------------------------------------ 1. exact reference, every family
@pytest.mark.parametrize("cfg", FAMILIES, ids=IDS)
def test_every_family_against_the_exact_reference(cfg):
    venv, inst = make_batch(cfg, 16, 31000)
    venv.reset()
    m = ge.MCTS(venv, 24)
    m.search(keyed_policy(m))
    torch.cuda.synchronize()
    assert int(m.visits[0].min()) == 25
    check_against_reference(m, venv, inst, cfg[0])
    assert int((m.visits[1:] > 0).sum()) > 16 * 4                 # simulations expanded nodes


@pytest.mark.parametrize("cfg", [FAMILIES[0], FAMILIES[7]], ids=[IDS[0], IDS[7]])
def test_bfloat16_logits_against_the_exact_reference(cfg):
    venv, inst = make_batch(cfg, 16, 32000)
    venv.reset()
    m = ge.MCTS(venv, 24, c_puct=0.75)
    m.search(keyed_policy(m, torch.bfloat16))       # ref_logits are multiples of 1/8 in [-1.75, 1.75]: exact in bfloat16
    torch.cuda.synchronize()
    check_against_reference(m, venv, inst, cfg[0], torch.bfloat16, c_puct=0.75)


# ------------------------------------------------------------------ 2. invariants and coverage on tiny instances
def all_prefixes(rep, limit):
    """Every action prefix of the oracle env from reset (the root excluded) and the best return of a finished episode, or None
    when there are more than `limit` prefixes."""
    out, best, stack = [], -math.inf, [()]
    while stack:
        p = stack.pop()
        mask, o, ret = rep(p)
        if p:
            out.append(p)
            if len(out) > limit:
                return None
            if o["done"]:
                best = max(best, ret)
                continue
        stack.extend(p + (int(a),) for a in np.flatnonzero(mask))
    return out, best


@pytest.mark.parametrize("tiny", TINY, ids=[t[0][:-3] for t in TINY])
def test_invariants_and_coverage_on_tiny_instances(tiny):
    env_id, N, E, kw = tiny
    probe = BatchedGraphEnv(env_id, 1, N, E, **kw)
    inst, reps, enum = [], [], []
    for s in range(300):                          # the first 6 seeds with at most 100 prefixes
        random.seed(s)
        np.random.seed(s)
        ins = generate_instance(env_id, probe.params)
        rep = Replayer(cu.oracle_from_instance(env_id, ins, probe.params))
        e = all_prefixes(rep, 100)
        if e is not None and e[1] > -math.inf:
            inst.append(ins)
            reps.append(rep)
            enum.append(e)
        if len(inst) == 6:
            break
    assert len(inst) == 6
    venv = BatchedGraphEnv(env_id, len(inst), N, E, **kw)
    venv.load_instances(inst)
    venv.reset()
    S = 2000
    m = ge.MCTS(venv, S, c_puct=4.0)
    m.search(keyed_policy(m, zero=True))
    torch.cuda.synchronize()
    for g in range(len(inst)):
        T = tree_of(m, g)
        rep, (prefixes, best) = reps[g], enum[g]
        assert int(T["visits"][0]) == S + 1
        seen = list(T["prefix"].values())
        assert len(seen) == len(set(seen)), "instance %d: a prefix appears twice" % g
        assert set(prefixes) <= set(seen), "instance %d: the tree does not hold every prefix" % g
        kids = {int(n): [] for n in T["created"]}
        for n in T["created"][1:]:
            kids[int(T["parent"][n])].append(int(n))
        best_tree = -math.inf
        for n in T["created"]:
            n = int(n)
            p = T["prefix"][n]
            mask, o, ret = rep(p)
            term = bool(T["terminal"][n])
            if n:
                assert term == bool(o["done"]) and _close(float(T["reward"][n]), o["reward"]), (g, p)
            total = sum(int(T["visits"][c]) for c in kids[n])
            if term or not mask.any():                # revisited: its own visits on top of its children's
                assert int(T["visits"][n]) >= 1 + total, (g, p)
            else:
                assert int(T["visits"][n]) == 1 + total, (g, p)
            if term:
                best_tree = max(best_tree, sum(float(T["reward"][c]) for c in _path(T, n)))
        assert _close(best_tree, best), g


def _path(T, n):
    out = []
    while n > 0:
        out.append(n)
        n = int(T["parent"][n])
    return out


# ------------------------------------------------------------------ 3. whole episodes
@pytest.mark.parametrize("cfg", [FAMILIES[0], FAMILIES[6], FAMILIES[10]], ids=[IDS[0], IDS[6], IDS[10]])
def test_run_replays_in_the_oracle(cfg):
    env_id = cfg[0]
    venv, inst = make_batch(cfg, 12, 33000)
    venv.reset()
    before = {k: v.clone() for k, v in venv.t.items()}
    m = ge.MCTS(venv, 16)
    pol = keyed_policy(m)
    m.search(pol)
    torch.cuda.synchronize()
    for k, v in venv.t.items():
        assert torch.equal(v, before[k]), "search() changed venv's %s" % k
    res = m.run(pol)
    assert res.found.any()
    for k, v in venv.t.items():
        assert torch.equal(v, before[k]), "run() changed venv's %s" % k
    acts = res.actions.cpu().numpy()
    for g in np.flatnonzero(res.found.cpu().numpy()):
        oe = cu.oracle_from_instance(env_id, inst[g], venv.params)
        r, o = 0.0, None
        for a in acts[g]:
            if a < 0:
                break
            assert o is None or not o["done"]
            o = oe.step(int(a))
            assert o["status"] == 0, (g, a)
            r += o["reward"]
        assert o["done"], g
        assert _close(res.ret[g].item(), r), g
        assert _close(res.solution_cost[g].item(), 0.0 if np.isnan(o["solution_cost"]) else o["solution_cost"]), g
        assert bool(res.solved[g]) == (o["solved"] == 1), g
        assert not math.isnan(res.root_value[g, 0].item())


def test_run_from_current_on_an_auto_reset_batch():
    venv, _ = make_batch(FAMILIES[0], 64, 34000)              # auto-reset on: some envs are on their second episode
    venv.enable_env_clock()
    venv.reset()
    for t in range(9):
        venv.step_sampled(5, t)
    before = {k: v.clone() for k, v in venv.t.items()}
    clock = venv.env_steps.clone()
    m = ge.MCTS(venv, 12)
    res = m.run(keyed_policy(m), from_current=True)
    for k, v in venv.t.items():
        assert torch.equal(v, before[k]), "venv's %s changed" % k
    assert torch.equal(venv.env_steps, clock)
    # the moves replayed from venv's current state on a device copy give the reported returns
    cp = venv.like(venv.B, auto_reset=False)
    cp.enable_env_clock()
    cp.gather_instances(venv)
    cp.load_states(venv.save_states())
    cp.t["acc"].zero_()
    for t in range(res.steps):
        cp.step(res.actions[:, t].contiguous())
    found = res.found
    assert found.any()
    assert torch.equal(cp.t["done"] != 0, found)
    assert torch.equal(cp.t["acc"][2][found], res.ret[found])


# ------------------------------------------------------------------ 4. edge cases
def test_one_simulation_and_done_roots():
    cfg = FAMILIES[1]                                         # ShortestPath N = 10
    venv, inst = make_batch(cfg, 32, 35000)
    venv.reset()
    m = ge.MCTS(venv, 1)
    m.search(keyed_policy(m))
    torch.cuda.synchronize()
    assert torch.equal(m.visits[0], torch.full_like(m.visits[0], 2))
    check_against_reference(m, venv, inst, cfg[0])
    # drive half the instances to the end of their episode (auto-reset off), then search from there
    env = venv.like(venv.B, auto_reset=False)
    env.gather_instances(venv)
    env.reset()
    for t in range(4 * venv.N):
        live = (env.t["done"] == 0) & (torch.arange(env.B, device="cuda") % 2 == 0)
        if not live.any():
            break
        a = env.sample_actions(7, t)
        env.step(torch.where(live, a, -1).int())
    done = env.t["done"] != 0
    assert done[::2].any() and not done[1::2].any()
    S = 6
    m2 = ge.MCTS(env, S)
    out = m2.search(keyed_policy(m2), env)
    torch.cuda.synchronize()
    d = done.nonzero().flatten()
    assert torch.equal(m2.visits[0], torch.full_like(m2.visits[0], S + 1))
    assert (m2.visits[0, d] == S + 1).all() and (m2.visits[1:, d] == 0).all()
    assert (m2.wsum[0, d] == 0).all() and (m2.terminal[0, d] == 1).all()
    assert (out.action[d] == -1).all() and (out.visits[d] == 0).all() and (out.value[d] == 0).all()
    assert torch.isnan(out.q[d]).all()
    assert (out.action[1::2] >= 0).all()


# ------------------------------------------------------------------ 5. scheduling
def _trees(m):
    return [x.clone() for x in (m.parent, m.action, m.visits, m.wsum.view(torch.int64), m.reward, m.value, m.terminal, m.mask,
                                m.qmin.view(torch.int64), m.qmax.view(torch.int64))]


def test_graph_replay_and_pdl_equal_eager():
    S = 20
    runs = {}
    for mode in ("eager", "graph", "pdl"):
        venv, inst = make_batch(FAMILIES[7], 40, 36000)     # Multicast, incremental masks
        venv.reset()
        m = ge.MCTS(venv, S)
        if mode == "pdl":
            m.leaf.enable_pdl()
        pol = keyed_policy(m)
        m.start(pol)
        if mode == "graph":
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                for _ in range(S):
                    m.simulate(pol)
            g.replay()
        else:
            for _ in range(S):
                m.simulate(pol)
        torch.cuda.synchronize()
        runs[mode] = _trees(m)
        if mode == "eager":
            check_against_reference(m, venv, inst, FAMILIES[7][0])
    for mode in ("graph", "pdl"):
        created = runs["eager"][2] > 0
        for i, (x, y) in enumerate(zip(runs["eager"], runs[mode])):
            sel = created if x.dim() == 2 else created[..., None].expand_as(x) if x.dim() == 3 else torch.ones_like(x, dtype=torch.bool)
            assert torch.equal(x[sel], y[sel]), "%s item %d" % (mode, i)
    assert int((runs["eager"][2][1:] > 0).sum()) > 40 * 10
