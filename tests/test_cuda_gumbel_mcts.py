"""GPU: Gumbel MuZero search (ge_gumbel_root / ge_gumbel_select / ge_gumbel_result, graphenvs_b200.GumbelMCTS).  Every kernel
family against a float64 restatement of include/graphenvs_b200.h, one simulation at a time; the root noise against its host
restatement, per seed, move and rank slice; one- and two-simulation searches sample the prior; sequential halving on tiny
instances; whole-episode decoding replayed in the oracle; CUDA-graph and PDL scheduling.  Fixed seeds: nothing here can flake."""
import math
import random
import sys

import numpy as np
import pytest
import torch
from scipy import stats

import cuda_util as cu
import graphenvs_b200 as ge
from graphenvs_b200 import BatchedGraphEnv
from graphenvs_b200.instances import generate_instance
from graphenvs_b200.mcts import considered_visits_table, unpack_mask
from test_cuda_beam import TINY
from test_cuda_env_state import FAMILIES, IDS, make_batch
from test_cuda_mcts import Replayer, _close, keyed_policy, ref_logits, ref_value
from test_cuda_stochastic_beam import gumbel64, mix32

pytestmark = pytest.mark.gpu

DBL_MIN = sys.float_info.min


# ------------------------------------------------------------------ the documented formulas, restated
def root_noise(seed, i, t, A):
    """node_gumbel(row_key(seed, i, t), a) for a in [0, A), in float64."""
    key = (mix32(seed, i, t) << np.uint64(32)) | mix32(np.uint64(seed) ^ np.uint64(0xD1B54A32D192ED03), i, t)
    return gumbel64(key, np.arange(A, dtype=np.uint64))


def lane_sum(items):
    """The kernels' fixed-order sum over (action, x) pairs in ascending action order: per lane a mod 32, then the butterfly."""
    part = [0.0] * 32
    for a, x in items:
        part[a % 32] = part[a % 32] + x
    for o in (16, 8, 4, 2, 1):
        part = [part[l] + part[l ^ o] for l in range(32)]
    return part[0]


def snapshot(m):
    """The device tree on the host; exp of the log-priors taken on the device (the kernels' float64 exp)."""
    T = {k: getattr(m, k).cpu().numpy() for k in ("parent", "action", "visits", "wsum", "reward", "value", "terminal", "child",
                                                  "prior")}
    T["mask"] = unpack_mask(m.mask, m.A).cpu().numpy()
    T["P"] = torch.exp(m.prior.double()).cpu().numpy()
    T["noise"] = m.noise.cpu().numpy()
    return T


def node_stats(T, g, s, vs, mi):
    """Completed Q at node s of instance g: (valid actions, N, child, q^, sigma, M)."""
    valid = np.flatnonzero(T["mask"][s, g]).tolist()
    N, C, Q = {}, {}, {}
    for a in valid:
        c = int(T["child"][s, g, a])
        n = int(T["visits"][c, g]) if c >= 0 else 0
        N[a], C[a] = n, c
        if n > 0:
            Q[a] = float(T["reward"][c, g]) + float(T["wsum"][c, g]) / n
    vis = [a for a in valid if N[a] > 0]
    P = {a: max(float(T["P"][s, g, a]), DBL_MIN) for a in vis}
    M = sum(N.values())
    maxn = max(N.values(), default=0)
    v = float(T["value"][s, g])
    if M:
        vmix = (v + M * (lane_sum((a, P[a] * Q[a]) for a in vis) / lane_sum((a, P[a]) for a in vis))) / (M + 1)
    else:
        vmix = v
    qh = {a: Q.get(a, vmix) for a in valid}
    lo, hi = min(qh.values(), default=0.0), max(qh.values(), default=0.0)
    den = max(hi - lo, 1e-8)
    cs = (mi + maxn) * vs
    sigma = {a: cs * ((qh[a] - lo) / den) for a in valid}
    return valid, N, C, qh, sigma, M


def softmax(T, g, s, valid, sigma):
    z = {a: float(T["prior"][s, g, a]) + sigma[a] for a in valid}
    zm = max(z.values())
    e = {a: math.exp(z[a] - zm) for a in valid}
    tot = math.fsum(e.values())
    return {a: e[a] / tot for a in valid}


def best_of(scores):
    """The arg-max of {action: score} with ties to the lowest action, and whether the top two are within 1e-9 relative."""
    order = sorted(scores, key=lambda a: (-scores[a], a))
    near = len(order) > 1 and abs(scores[order[0]] - scores[order[1]]) <= 1e-9 * max(abs(scores[order[0]]), abs(scores[order[1]]))
    return order[0], near


def reference_select(T, g, S, m, vs, mi, table):
    """Selection of include/graphenvs_b200.h on the snapshot: (node, action, depth, near-tie seen, interior scores by node)."""
    s, depth, near_any, interior = 0, 0, False, {}
    while not T["terminal"][s, g]:
        valid, N, C, qh, sigma, M = node_stats(T, g, s, vs, mi)
        if not valid:
            break
        if s == 0:
            vstar = table[min(m, len(valid))][min(M, S - 1)]
            sc = {a: (float(T["noise"][g, a]) + float(T["prior"][0, g, a])) + sigma[a] for a in valid if N[a] == vstar}
            if not sc:
                break
            a, _ = best_of(sc)
        else:
            pi = softmax(T, g, s, valid, sigma)
            sc = {a: pi[a] - N[a] / (1 + M) for a in valid}
            a, near = best_of(sc)
            interior[s] = sc
            near_any |= near
        depth += 1
        if C[a] < 0:
            return s, a, depth, near_any, interior
        s = C[a]
    return s, -1, depth, near_any, interior


def reference_readout(T, g, m, vs, mi):
    valid, N, C, qh, sigma, M = node_stats(T, g, 0, vs, mi)
    pol = np.zeros(T["mask"].shape[-1])
    cq = np.full(T["mask"].shape[-1], np.nan)
    if valid:
        pi = softmax(T, g, 0, valid, sigma)
        for a in valid:
            pol[a], cq[a] = pi[a], qh[a]
    maxn = max(N.values(), default=0)
    sc = {a: (float(T["noise"][g, a]) + float(T["prior"][0, g, a])) + sigma[a] for a in valid if N[a] == maxn}
    action = -1 if T["terminal"][0, g] or not sc else best_of(sc)[0]
    return action, pol, cq, min(m, len(valid))


# ------------------------------------------------------------------ 1. every family, one simulation at a time
def replay_tree(G, S, sels, T_final, venv, g):
    """The tree of instance g rebuilt from the device's selections with the header's expansion and backup (r, terminal from
    the device, v from the keyed policy): (parent, action, N, Wsum) per created node."""
    nodes = {0: dict(parent=-1, action=-1, depth=0, N=0, W=0.0)}

    def r_of(n):
        return float(T_final["reward"][n, g])

    def v_of(n):
        return 0.0 if T_final["terminal"][n, g] else ref_value(g, nodes[n]["depth"], nodes[n]["action"])

    def backup(n):
        ret = v_of(n)
        while True:
            nd = nodes[n]
            nd["N"] += 1
            nd["W"] = nd["W"] + ret
            if n == 0:
                return
            ret = r_of(n) + ret
            n = nd["parent"]

    backup(0)
    for k in range(1, S + 1):
        s, a = sels[k - 1][0][g], sels[k - 1][1][g]
        if a >= 0:
            nodes[k] = dict(parent=int(s), action=int(a), depth=nodes[int(s)]["depth"] + 1, N=0, W=0.0)
            backup(k)
        else:
            backup(int(s))
    return nodes


def run_checked(m, venv, inst, env_id, pol, t=0, dtype=torch.float32):
    """A whole search with the restatement's selection checked after every simulation; returns the number of near ties."""
    G, S, A = m.G, m.S, m.A
    table = considered_visits_table(m.max_considered, S)
    m.start(pol, t=t)
    sels, near_ties = [], 0
    for k in range(1, S + 1):
        T = snapshot(m)
        m.simulate(pol)
        sel = (m.sel_node.cpu().numpy(), m.sel_action.cpu().numpy(), m.depth.cpu().numpy())
        sels.append(sel)
        for g in range(G):
            s, a, d, near, _ = reference_select(T, g, S, m.max_considered, m.value_scale, m.maxvisit_init, table)
            got = (int(sel[0][g]), int(sel[1][g]), int(sel[2][g]))
            if got != (s, a, d):
                assert near, "simulation %d instance %d: device %s, restatement %s" % (k, g, got, (s, a, d))
                near_ties += 1
    out = m.result()
    torch.cuda.synchronize()
    T = snapshot(m)
    for g in range(G):
        rep = Replayer(cu.oracle_from_instance(env_id, inst[g], venv.params))
        nodes = replay_tree(G, S, sels, T, venv, g)
        created = np.flatnonzero(T["visits"][:, g] > 0).tolist()
        assert created == sorted(nodes), "instance %d: created nodes" % g
        prefix = {0: ()}
        for n in sorted(nodes):
            nd = nodes[n]
            tag = "instance %d node %d" % (g, n)
            assert int(T["parent"][n, g]) == nd["parent"] and int(T["action"][n, g]) == nd["action"], tag
            assert int(T["visits"][n, g]) == nd["N"], tag
            assert float(T["wsum"][n, g]) == nd["W"], tag                       # bit for bit
            if n:
                prefix[n] = prefix[nd["parent"]] + (nd["action"],)
            mask, o, _ = rep(prefix[n])
            term = bool(o["done"]) if n else bool(venv.t["done"][g].item())
            assert bool(T["terminal"][n, g]) == term, tag
            if n:
                assert _close(float(T["reward"][n, g]), o["reward"]), tag
            if term:
                continue
            assert np.array_equal(T["mask"][n, g], mask), tag
            lg = torch.from_numpy(ref_logits(g, len(prefix[n]), nd["action"], A)).to(dtype).double()
            lg[~torch.from_numpy(mask)] = -math.inf
            lsm = torch.log_softmax(lg, 0).numpy()
            np.testing.assert_allclose(T["prior"][n, g][mask], lsm[mask], rtol=1e-6, atol=2e-6, err_msg=tag)
        action, pol_ref, cq, considered = reference_readout(T, g, m.max_considered, m.value_scale, m.maxvisit_init)
        assert int(out.action[g]) == action, g
        q = out.completed_q[g].cpu().numpy()
        assert np.array_equal(np.isnan(q), np.isnan(cq)) and np.array_equal(q[~np.isnan(q)], cq[~np.isnan(cq)]), g   # exact
        np.testing.assert_allclose(out.policy[g].cpu().numpy(), pol_ref, rtol=0, atol=1e-6)
        assert int(out.considered[g]) == considered
        ch = T["child"][0, g]
        want = [nodes[int(ch[a])]["N"] if T["mask"][0, g, a] and ch[a] >= 0 else 0 for a in range(A)]
        assert out.visits[g].cpu().tolist() == want, g
    return near_ties


@pytest.mark.parametrize("cfg", FAMILIES, ids=IDS)
def test_every_family_against_the_restatement(cfg):
    venv, inst = make_batch(cfg, 16, 41000)
    venv.reset()
    m = ge.GumbelMCTS(venv, 24, max_considered=8, seed=5)
    near = run_checked(m, venv, inst, cfg[0], keyed_policy(m))
    print("near ties:", near)
    assert near <= 2
    assert int(m.visits[0].min()) == 25
    assert int((m.visits[1:] > 0).sum()) > 16 * 4


@pytest.mark.parametrize("cfg", [FAMILIES[0], FAMILIES[7]], ids=[IDS[0], IDS[7]])
def test_bfloat16_logits_against_the_restatement(cfg):
    venv, inst = make_batch(cfg, 16, 42000)
    venv.reset()
    m = ge.GumbelMCTS(venv, 24, max_considered=4, value_scale=0.3, maxvisit_init=10.0, seed=6)
    near = run_checked(m, venv, inst, cfg[0], keyed_policy(m, torch.bfloat16), t=3, dtype=torch.bfloat16)
    print("near ties:", near)
    assert near <= 2


# ------------------------------------------------------------------ 2. root noise
def test_root_noise_seed_move_and_rank_slice():
    cfg = FAMILIES[2]                                        # MaxIndependentSet N = 50: every node valid at the root
    venv, _ = make_batch(cfg, 64, 43000)
    venv.reset()
    m = ge.GumbelMCTS(venv, 8, seed=123)
    pol = keyed_policy(m)
    out = m.search(pol, t=4)
    torch.cuda.synchronize()
    mask = unpack_mask(m.mask[0], m.A).cpu().numpy()
    noise = m.noise.cpu().numpy()
    for g in range(m.G):
        ref = root_noise(123, g, 4, m.A)
        d = noise[g][mask[g]].astype(np.float64)
        assert np.all(np.abs(d - ref[mask[g]]) <= 4 * 2.0 ** -23 * (1 + np.abs(ref[mask[g]]))), g
        assert np.all(noise[g][~mask[g]] == 0), g            # written under the root's mask only
    keep = [x.clone() for x in (m.noise, m.visits, m.parent, m.action, m.wsum, out.action, out.policy)]
    again = m.search(pol, t=4)
    for x, y in zip(keep, (m.noise, m.visits, m.parent, m.action, m.wsum, again.action, again.policy)):
        assert torch.equal(x, y)
    m.search(pol, t=5)
    sel = torch.from_numpy(mask).cuda()
    assert not torch.equal(m.noise[sel], keep[0][sel])
    # instances [16, 48) searched on their own with env_id0 = 16 and a policy keyed by the global instance id
    lo, n = 16, 32
    full, _ = make_batch(cfg, 64, 43000)
    part, _ = make_batch(cfg, n, 43000 + lo, env_id0=lo)
    res = {}
    for name, env, off in (("full", full, 0), ("part", part, lo)):
        env.reset()
        mm = ge.GumbelMCTS(env, 12, max_considered=4, seed=77)
        res[name] = (mm.search(global_keyed(mm, off), t=2), [x.clone() for x in (mm.noise, mm.visits, mm.parent, mm.action,
                                                                               mm.wsum, mm.sel_node)])
    (fo, ft), (po, pt) = res["full"], res["part"]
    for k in ("action", "policy", "completed_q", "visits", "considered"):
        x, y = getattr(fo, k)[lo:lo + n], getattr(po, k)
        if x.is_floating_point():
            assert torch.equal(x.isnan(), y.isnan()) and torch.equal(torch.nan_to_num(x, 7.0), torch.nan_to_num(y, 7.0)), k
        else:
            assert torch.equal(x, y), k
    assert torch.equal(ft[0][lo:lo + n], pt[0]) and torch.equal(ft[5][lo:lo + n], pt[5])   # noise [G, A], sel_node [G]
    for x, y in zip(ft[1:5], pt[1:5]):                                                       # per node [S + 1, G]
        assert torch.equal(x[:, lo:lo + n], y)


def global_keyed(m, off):
    """keyed_policy with the instance index offset by `off` (the global instance id of a rank slice)."""
    G, A = m.G, m.A
    g = off + torch.arange(G, device="cuda", dtype=torch.int64)
    a = torch.arange(A, device="cuda", dtype=torch.int64)

    def policy(env):
        k = (g * 131 + m.depth.long() * 17 + (m.sel_action.long() + 1) * 7)[:, None]
        logits = (((k * 37 + a * 11 + (k * a) % 23) % 29 - 14).float() * 0.125)
        value = ((k[:, 0] * 13) % 41 - 20).float() / 8
        return logits, value
    return policy


# ------------------------------------------------------------------ 3. with value_scale = 0 and S = m <= 2 the action samples the prior
@pytest.mark.parametrize("S", [1, 2])
def test_one_and_two_simulations_sample_the_prior(S):
    env_id, N, E, kw, _ = FAMILIES[2]                       # MaxIndependentSet N = 50
    one, _ = make_batch(FAMILIES[2], 1, 44000)
    Gn = 16384
    venv = BatchedGraphEnv(env_id, Gn, N, E, **kw)
    venv.gather_instances(one, torch.zeros(Gn, dtype=torch.int32, device="cuda"))
    venv.reset()
    A = venv.desc.A
    gen = torch.Generator(device="cuda").manual_seed(8)
    m = ge.GumbelMCTS(venv, S, max_considered=S, value_scale=0.0, seed=2024)
    for row in range(3):
        lg = torch.randn(A, generator=gen, device="cuda") * 1.2
        pol = lambda env: (lg.expand(Gn, A).contiguous(), torch.zeros(Gn, device="cuda"))   # noqa: E731
        out = m.search(pol, t=row)
        valid = unpack_mask(m.mask[0, 0], A).cpu().numpy()
        assert valid.sum() >= 10
        lp = m.prior[0, 0].double().cpu().numpy()
        p = np.exp(lp[valid])
        p /= p.sum()
        acts = out.action.cpu().numpy()
        assert (acts >= 0).all() and valid[acts].all()
        counts = np.bincount(acts, minlength=A)[valid]
        exp = Gn * p
        small = exp < 5                                     # pooled into one bin
        obs = np.append(counts[~small], counts[small].sum())
        ex = np.append(exp[~small], exp[small].sum())
        chi2 = ((obs - ex) ** 2 / np.maximum(ex, 1e-12)).sum()
        dof = int((~small).sum()) + (1 if small.any() else 0) - 1
        assert stats.chi2.sf(chi2, dof) > 1e-6, (row, counts, exp)


# ------------------------------------------------------------------ 4. sequential halving on tiny instances
def halving_multiset(row):
    """The visit counts the table row prescribes: step j visits an action with count row[j]."""
    counts = []
    for v in row:
        i = counts.index(v) if v in counts else None
        if i is None:
            assert v == 0
            counts.append(1)
        else:
            counts[i] += 1
    return sorted(counts, reverse=True)


@pytest.mark.parametrize("mc", [2, 4, 16])
@pytest.mark.parametrize("tiny", TINY, ids=[t[0][:-3] for t in TINY])
def test_sequential_halving_on_tiny_instances(tiny, mc):
    env_id, N, E, kw = tiny
    probe = BatchedGraphEnv(env_id, 1, N, E, **kw)
    inst = []
    for s in range(8):
        random.seed(s)
        np.random.seed(s)
        inst.append(generate_instance(env_id, probe.params))
    venv = BatchedGraphEnv(env_id, len(inst), N, E, **kw)
    venv.load_instances(inst)
    venv.reset()
    S = 32
    m = ge.GumbelMCTS(venv, S, max_considered=mc, seed=9)
    out = m.search(keyed_policy(m), t=1)
    torch.cuda.synchronize()
    table = considered_visits_table(mc, S)
    visits, valid = out.visits.cpu().numpy(), unpack_mask(m.mask[0], m.A).cpu().numpy()
    pol = out.policy.cpu().numpy()
    for g in range(len(inst)):
        assert int(m.visits[0, g]) == S + 1
        if not valid[g].any():
            continue
        mp = min(mc, int(valid[g].sum()))
        assert int(out.considered[g]) == mp
        want = halving_multiset(table[mp])
        got = sorted((int(x) for x in visits[g][valid[g]] if x > 0), reverse=True)
        assert got == want, (g, mp, got, want)
        assert abs(pol[g].sum() - 1.0) < 1e-5 and np.all(pol[g][~valid[g]] == 0)
        a = int(out.action[g])
        assert valid[g][a] and visits[g][a] == visits[g].max(), g


# ------------------------------------------------------------------ 5. whole episodes
@pytest.mark.parametrize("cfg", [FAMILIES[0], FAMILIES[6], FAMILIES[10]], ids=[IDS[0], IDS[6], IDS[10]])
def test_run_replays_in_the_oracle(cfg):
    env_id = cfg[0]
    venv, inst = make_batch(cfg, 12, 45000)
    venv.reset()
    before = {k: v.clone() for k, v in venv.t.items()}
    m = ge.GumbelMCTS(venv, 8, max_considered=4, seed=3)
    pol = keyed_policy(m)
    res = m.run(pol)
    for k, v in venv.t.items():
        assert torch.equal(v, before[k]), "run() changed venv's %s" % k
    assert res.found.any()
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


# ------------------------------------------------------------------ 6. scheduling
def test_graph_replay_and_pdl_equal_eager():
    S = 20
    runs = {}
    for mode in ("eager", "graph", "pdl"):
        venv, inst = make_batch(FAMILIES[7], 40, 46000)     # Multicast, incremental masks
        venv.reset()
        m = ge.GumbelMCTS(venv, S, max_considered=8, seed=11)
        if mode == "pdl":
            m.leaf.enable_pdl()
        pol = keyed_policy(m)
        m.start(pol, t=1)
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
        out = m.result()
        torch.cuda.synchronize()
        runs[mode] = [x.clone() for x in (m.parent, m.action, m.visits, m.wsum.view(torch.int64), m.reward, m.value, m.terminal,
                                          m.mask, m.noise, out.action, out.policy, out.completed_q.view(torch.int64))]
    for mode in ("graph", "pdl"):
        created = runs["eager"][2] > 0
        for i, (x, y) in enumerate(zip(runs["eager"], runs[mode])):
            sel = created if i < 7 else created[..., None].expand_as(x) if i == 7 else torch.ones_like(x, dtype=torch.bool)
            assert torch.equal(x[sel], y[sel]), "%s item %d" % (mode, i)
    assert int((runs["eager"][2][1:] > 0).sum()) > 40 * 10
