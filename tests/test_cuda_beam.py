"""GPU: beam search (ge_beam_expand, graphenvs_b200.BeamSearch).  The expand kernel against an exact numpy reference bit for
bit; width 1 against the greedy rollout in every kernel family; exhaustive search on tiny instances against the C oracle's
enumeration; every family at W = 8 against the oracle and the masked log-probs along each beam; decoding from a mid-episode
state; and slice / CUDA-graph / PDL scheduling."""
import ctypes as C
import random

import numpy as np
import pytest
import torch

import cuda_util as cu
import graphenvs_b200 as ge
from graphenvs_b200 import BatchedGraphEnv, _native, policy as pol
from graphenvs_b200.instances import generate_instance
from test_cuda_env_state import FAMILIES, IDS, make_batch

pytestmark = pytest.mark.gpu

NEG = float("-inf")


def _p(t):
    return C.c_void_p(t.data_ptr())


def same(x, y):
    return torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x, y.view(torch.int32) if y.dtype == torch.float32 else y)


# ------------------------------------------------------------------ 1. the kernel against an exact reference
def _dummy_desc(B, A, mask, done):
    d = _native.GeBatch()
    if A == 8000:
        d.kind, d.N, d.M = 6, 500, 8000          # edge actions: A = M
    else:
        d.kind, d.N, d.M = 1, A, 2 * A           # node actions: A = N
    d.B = B
    assert _native.lib().ge_fill_layout(C.byref(d)) == 0 and d.A == A
    d.mask_bits, d.done = mask.data_ptr(), done.data_ptr()
    return d


def _expand(d, W, logits, score, dev="cuda"):
    B = d.B
    out = [torch.full((B,), 7.0, device=dev)] + [torch.full((B,), 7, dtype=torch.int32, device=dev) for _ in range(3)]
    _native.check(_native.lib().ge_beam_expand(C.byref(d), W, _p(logits), pol._DTYPES[logits.dtype], _p(score), *[_p(t) for t in out],
                                               C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out


def reference_expand(logits, valid, done, score, W):
    """Exact reference: log-probs from masked_log_prob (lse of the native forward, then fl32(l - lse), checked against
    masked_log_prob on sampled pairs), fl32 sums in torch, a stable lexsort in numpy by (score desc, parent, action)."""
    B, A = logits.shape
    AW = (A + 31) // 32
    packed = np.packbits(np.pad(valid, ((0, 0), (0, AW * 32 - A))), axis=1, bitorder="little").view(np.int32)
    mb = torch.from_numpy(packed.copy()).cuda()
    lp, ent, lse = (torch.empty(B, device="cuda") for _ in range(3))
    acts = torch.zeros(B, dtype=torch.int32, device="cuda")
    _native.check(_native.lib().ge_masked_log_prob(_p(logits), pol._DTYPES[logits.dtype], B, A, _p(mb), _p(acts), _p(lp), _p(ent), _p(lse), None))
    lpa = logits.float() - lse[:, None]                                   # fl32(l_a - lse) at every valid (row, action)
    r, a = np.nonzero(valid)
    if r.size:
        k = np.random.default_rng(0).choice(r.size, size=min(r.size, 4096), replace=False)
        rr, aa = torch.from_numpy(r[k]).cuda(), torch.from_numpy(a[k]).cuda()
        lp_s, _ = ge.masked_log_prob(logits[rr], mb[rr], aa.int())
        assert same(lp_s, lpa[rr, aa])
    sc = (torch.from_numpy(score).cuda()[:, None] + lpa).cpu().numpy()   # fl32(score + lp)
    exp = {k: np.empty(B, dt) for k, dt in (("parent", np.int32), ("action", np.int32), ("score", np.float32), ("load", np.int32))}
    for g in range(B // W):
        rows = range(g * W, g * W + W)
        cs, cp, ca = [], [], []
        for b in rows:
            if score[b] == NEG:
                continue
            if done[b]:
                cs.append(np.float32(score[b])); cp.append(b); ca.append(-1)
                continue
            av = np.flatnonzero(valid[b])
            cs.extend(sc[b, av]); cp.extend([b] * av.size); ca.extend(av.tolist())
        cs, cp, ca = np.array(cs, np.float32), np.array(cp, np.int64), np.array(ca, np.int64)
        order = np.lexsort((ca, cp, -cs))[:W]
        for j, b in enumerate(rows):
            if j < order.size:
                o = order[j]
                exp["parent"][b], exp["action"][b], exp["score"][b] = cp[o], ca[o], cs[o]
                exp["load"][b] = -1 if cp[o] == b else cp[o]
            else:
                exp["parent"][b], exp["action"][b], exp["score"][b], exp["load"][b] = -1, -1, NEG, -1
    return exp


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("A", [7, 50, 200, 8000])
@pytest.mark.parametrize("W", [1, 2, 5, 16, 32])
def test_expand_equals_exact_reference(W, A, dtype):
    rng = np.random.default_rng(W * 100003 + A + (dtype == torch.bfloat16))
    G = max(2, 160 // W)
    B = G * W
    vals = rng.integers(-3, 2, size=(B, A)).astype(np.float32) * 0.5    # few values: ties are common
    density = rng.choice([0.0, 0.03, 0.3, 1.0], size=B)
    valid = rng.random((B, A)) < density[:, None]
    done = rng.random(B) < 0.2
    score = (-rng.integers(0, 3, size=B) * 0.25).astype(np.float32)
    score[rng.random(B) < 0.2] = NEG
    score[::W] = np.where(rng.random(B // W) < 0.5, 0.0, score[::W])
    vals[~valid] = np.nan                                                # invalid logits are never read
    logits = torch.from_numpy(vals).cuda().to(dtype)
    AW = (A + 31) // 32
    packed = np.packbits(np.pad(valid, ((0, 0), (0, AW * 32 - A))), axis=1, bitorder="little").view(np.uint32).copy()
    if A % 32:
        packed[:, -1] |= np.uint32(0xFFFFFFFF) << np.uint32(A % 32)     # stray bits past A are ignored
    mask = torch.from_numpy(packed.view(np.int32)).cuda()
    done_t = torch.from_numpy(done.astype(np.uint8)).cuda()
    d = _dummy_desc(B, A, mask, done_t)
    exp = reference_expand(logits, valid, done, score, W)
    score_t = torch.from_numpy(score).cuda()
    so, par, act, load = _expand(d, W, logits, score_t)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(par.cpu().numpy(), exp["parent"])
    np.testing.assert_array_equal(act.cpu().numpy(), exp["action"])
    np.testing.assert_array_equal(so.cpu().numpy().view(np.int32), exp["score"].view(np.int32))
    np.testing.assert_array_equal(load.cpu().numpy(), exp["load"])
    # deterministic
    again = _expand(d, W, logits, score_t)
    assert all(same(x, y) for x, y in zip(again, (so, par, act, load)))


# ------------------------------------------------------------------ policies
def table_policy(venv, W, scale=1.0, seed=0, separated=False):
    """logits of wide env b = table[instance b // W, head b, :]: state-dependent through the head.  separated=True: every row
    is a permutation of 0 .. A-1, so valid logits differ by at least 1 (greedy and width-1 beam then agree)."""
    G, N, A = venv.B, venv.N, venv.desc.A
    gen = torch.Generator(device="cuda").manual_seed(seed)
    if separated:
        tab = torch.argsort(torch.rand((G, N, A), generator=gen, device="cuda"), dim=-1).float()
    else:
        tab = torch.randn((G, N, A), generator=gen, device="cuda") * scale
    cache = {}

    def policy(env):
        if env.B not in cache:
            cache[env.B] = torch.arange(env.B, device="cuda") // (env.B // G)
        inst = cache[env.B]
        return tab[inst, env.t["head"].long().clamp(0, N - 1)]
    return policy


def greedy_rollout(venv, policy, from_current=False, max_steps=None):
    """The greedy rollout of every instance of venv (a copy, auto-reset off): per env its actions until done, and acc."""
    ref = venv.like(venv.B, auto_reset=False)
    if venv.env_steps is not None:
        ref.enable_env_clock()
    ref.gather_instances(venv)
    if from_current:
        ref.load_states(venv.save_states())
    else:
        ref.reset()
    ref.t["acc"].zero_()
    T = max_steps or 4 * venv.N
    seqs = [[] for _ in range(venv.B)]
    for t in range(T):
        done = ref.t["done"].cpu().numpy().astype(bool)
        if done.all():
            break
        acts, _, _ = ref.sample_logits(policy(ref), 0, t, greedy=True)
        a = acts.cpu().numpy()
        for b in np.flatnonzero(~done):
            seqs[b].append(int(a[b]))
        ref.step(acts)
    torch.cuda.synchronize()
    return seqs, ref.t["acc"].clone(), ref.t["done"].clone()


def trim(row):
    row = [int(x) for x in row]
    while row and row[-1] == -1:
        row.pop()
    return row


# ------------------------------------------------------------------ 2. width 1 is greedy
@pytest.mark.parametrize("cfg", FAMILIES, ids=IDS)
def test_width_one_equals_greedy(cfg):
    venv, _ = make_batch(cfg, 40, 9100)
    pol_fn = table_policy(venv, 1, seed=3, separated=True)
    seqs, acc, done = greedy_rollout(venv, pol_fn)
    res = ge.BeamSearch(venv, width=1).run(pol_fn)
    d = done.cpu().numpy().astype(bool)
    assert d.any() or cfg[0] == "PerishableProductDelivery-v0"     # (a head-indexed greedy courier can circle until the cap)
    for g in range(venv.B):
        assert bool(res.found[g]) == d[g], g
        beam = trim(res.beams.actions[g, 0].cpu().numpy())
        assert beam == seqs[g], "instance %d" % g
        if d[g]:
            assert trim(res.actions[g].cpu().numpy()) == seqs[g]
            assert res.ret[g].item() == acc[2, g].item() and bool(res.solved[g]) == (acc[1, g].item() > 0)


# ------------------------------------------------------------------ 3. exhaustive on tiny instances
TINY = [("ShortestPath-v0", 8, 10, {}), ("LongestPath-v0", 8, 10, {"parenting": 2}), ("TSP-v0", 5, 8, {"parenting": 1}),
        ("MaxIndependentSet-v0", 4, 4, {}), ("SteinerTree-v0", 5, 5, {"n_dests": 2})]


def enumerate_trajectories(oe, W):
    """Every complete trajectory of the oracle env from reset (each prefix replayed from reset) with its last step's outputs,
    or None when a beam of width W cannot hold the prefix tree (live prefixes + finished trajectories > W at some depth)."""
    def replay(prefix):
        oe.reset_state()
        m, o, ret = oe.mask(reset_patch=True), None, 0.0
        for a in prefix:
            o = oe.step(a)
            ret += o["reward"]
            if o["has_mask"]:
                m = o["mask"]
        return m, o, ret
    live, finished = [()], {}
    while live:
        nxt = []
        for p in live:
            m, _, _ = replay(p)
            for a in np.flatnonzero(m):
                q = p + (int(a),)
                _, o, ret = replay(q)
                if o["done"]:
                    finished[q] = (ret, o)
                else:
                    nxt.append(q)
        if len(nxt) + len(finished) > W:
            return None
        live = nxt
    return finished


def _close(x, y):
    return abs(x - y) <= 1e-5 * max(1.0, abs(y))


@pytest.mark.parametrize("tiny", TINY, ids=[t[0][:-3] for t in TINY])
def test_exhaustive_on_tiny_instances(tiny):
    env_id, N, E, kw = tiny
    W = 32
    probe = BatchedGraphEnv(env_id, 1, N, E, **kw)
    inst, trees = [], []
    for s in range(200):                         # the first 6 seeds whose prefix tree fits a beam of width 32
        random.seed(s)
        np.random.seed(s)
        ins = generate_instance(env_id, probe.params)
        tree = enumerate_trajectories(cu.oracle_from_instance(env_id, ins, probe.params), W)
        if tree is not None:
            inst.append(ins)
            trees.append(tree)
        if len(inst) == 6:
            break
    assert len(inst) == 6
    venv = BatchedGraphEnv(env_id, len(inst), N, E, **kw)
    venv.load_instances(inst)
    res = ge.BeamSearch(venv, width=W).run(lambda env: torch.zeros((env.B, env.desc.A), device="cuda"))
    for g, tree in enumerate(trees):
        alive = (res.beams.score[g] > NEG).cpu().numpy()
        done = res.beams.done[g].cpu().numpy()
        got = {}
        for j in np.flatnonzero(alive):
            assert done[j], "instance %d slot %d did not finish" % (g, j)
            got[tuple(trim(res.beams.actions[g, j].cpu().numpy()))] = j
        assert set(got) == set(tree), "instance %d" % g
        for q, j in got.items():
            ret, o = tree[q]
            assert _close(res.beams.ret[g, j].item(), ret), (g, q)
            sol = 0.0 if np.isnan(o["solution_cost"]) else o["solution_cost"]
            assert _close(res.beams.solution_cost[g, j].item(), sol), (g, q)
            assert bool(res.beams.solved[g, j]) == (o["solved"] == 1), (g, q)
        best = max(r for r, _ in tree.values())
        assert bool(res.found[g]) and _close(res.ret[g].item(), best)


# ------------------------------------------------------------------ 4. every family at W = 8 against the oracle
def replay_scores(venv, W, policy, actions):
    """Replays every beam's sequence in a fresh wide batch: the fl32 sum of masked_log_prob terms and acc per env."""
    rep = venv.like(venv.B * W, auto_reset=False)
    rep.gather_instances(venv, torch.arange(venv.B, dtype=torch.int32, device="cuda").repeat_interleave(W))
    rep.reset()
    rep.t["acc"].zero_()
    B, T = rep.B, actions.shape[-1]
    acts = actions.reshape(B, T)
    s = torch.zeros(B, device="cuda")
    for t in range(T):
        a = acts[:, t].contiguous()
        lp, _ = ge.masked_log_prob(policy(rep), rep.t["mask_bits"], a)
        s = torch.where(a >= 0, s + lp, s)
        rep.step(a)
    return s, rep.t["acc"]


@pytest.mark.parametrize("cfg", FAMILIES, ids=IDS)
def test_every_family_against_the_oracle(cfg):
    env_id = cfg[0]
    W, G = 8, 200
    venv, inst = make_batch(cfg, G, 12000)
    pol_fn = table_policy(venv, W, scale=2.0, seed=11)
    res = ge.BeamSearch(venv, width=W).run(pol_fn)
    found = res.found.cpu().numpy()
    assert found.any() or env_id == "PerishableProductDelivery-v0"
    alive = res.beams.score > NEG
    s, acc = replay_scores(venv, W, pol_fn, torch.where(alive[..., None], res.beams.actions, -1))
    a = alive.flatten()
    assert same(s[a], res.beams.score.flatten()[a]), "beam scores are the sums of masked_log_prob terms"
    assert torch.equal(acc[2][a], res.beams.ret.flatten()[a])
    acts, ret, cost, solved = res.actions.cpu().numpy(), res.ret.cpu().numpy(), res.solution_cost.cpu().numpy(), res.solved.cpu().numpy()
    for g in np.flatnonzero(found):
        oe = cu.oracle_from_instance(env_id, inst[g], venv.params)
        r, o = 0.0, None
        for x in trim(acts[g]):
            assert o is None or not o["done"]
            o = oe.step(x)
            assert o["status"] == 0, (g, x)
            r += o["reward"]
        assert o["done"], g
        tag = "%s instance %d" % (env_id, g)
        assert _close(ret[g], r), tag
        assert _close(cost[g], 0.0 if np.isnan(o["solution_cost"]) else o["solution_cost"]), tag
        assert bool(solved[g]) == (o["solved"] == 1), tag


# ------------------------------------------------------------------ 5. decoding from the current state
@pytest.mark.parametrize("cfg", [FAMILIES[0], FAMILIES[6]], ids=[IDS[0], IDS[6]])
def test_from_current_continues_like_greedy(cfg):
    venv, _ = make_batch(cfg, 64, 15000)                  # auto-reset on: some envs are on their second episode
    venv.reset()
    for t in range(7):
        venv.step_sampled(5, t)
    before = {k: v.clone() for k, v in venv.t.items()}
    pol_fn = table_policy(venv, 1, seed=8, separated=True)
    seqs, acc, done = greedy_rollout(venv, pol_fn, from_current=True)
    res = ge.BeamSearch(venv, width=1).run(pol_fn, from_current=True)
    for k, v in venv.t.items():
        assert torch.equal(v, before[k]), "venv's %s changed" % k
    d = done.cpu().numpy().astype(bool)
    for g in range(venv.B):
        assert trim(res.beams.actions[g, 0].cpu().numpy()) == seqs[g], g
        assert bool(res.found[g]) == d[g]
        if d[g]:
            assert res.ret[g].item() == acc[2, g].item()


# ------------------------------------------------------------------ 6. scheduling
def _sched_bs(pdl=False):
    venv = BatchedGraphEnv("LongestPath-v0", 128, 50, 200, parenting=2, auto_reset=True)
    venv.generate(seed=23)
    bs = ge.BeamSearch(venv, width=8)
    if pdl:
        bs.wide.enable_pdl()
    return venv, bs


def test_graph_replay_and_pdl_equal_eager():
    T = 12
    runs = {}
    for mode in ("eager", "graph", "pdl"):
        venv, bs = _sched_bs(pdl=mode == "pdl")
        pol_fn = table_policy(venv, 8, scale=0.5, seed=4)
        bs.start()
        bs.reserve(T)
        if mode == "graph":
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                for _ in range(T):
                    bs.advance(pol_fn(bs.wide))
            g.replay()
        else:
            for _ in range(T):
                bs.advance(pol_fn(bs.wide))
        torch.cuda.synchronize()
        runs[mode] = (bs._parents[:T].clone(), bs._actions[:T].clone(), bs.score.clone(), bs.wide.t["acc"].clone(),
                      bs.wide.t["traj"].clone(), bs.wide.t["mask_bits"].clone(), bs.wide.t["done"].clone())
    for mode in ("graph", "pdl"):
        for i, (x, y) in enumerate(zip(runs["eager"], runs[mode])):
            assert same(x, y), "%s item %d" % (mode, i)
    assert (runs["eager"][1][1:] >= 0).any() and (runs["eager"][0][1] != torch.arange(1024, device="cuda")).any()


def test_expand_over_slices_equals_one_descriptor():
    venv, bs = _sched_bs()
    pol_fn = table_policy(venv, 8, scale=0.5, seed=5)
    bs.start()
    for _ in range(4):
        bs.advance(pol_fn(bs.wide))
    wide = bs.wide
    logits = pol_fn(wide).to(torch.bfloat16).contiguous()
    full = _expand(wide.desc, 8, logits, bs.score)
    B, lo = wide.B, 512
    parts = [torch.full((B,), 7.0, device="cuda")] + [torch.full((B,), 7, dtype=torch.int32, device="cuda") for _ in range(3)]
    L = wide.lib
    for start, n in ((0, lo), (lo, B - lo)):
        d = wide.slice_desc(start, n)
        _native.check(L.ge_beam_expand(C.byref(d), 8, _p(logits[start:]), pol._DTYPES[logits.dtype], _p(bs.score[start:]),
                                       *[_p(t[start:]) for t in parts], wide._stream()))
    torch.cuda.synchronize()
    so, par, act, load = parts
    off = torch.zeros(B, dtype=torch.int32, device="cuda")
    off[lo:] = lo                                           # indices of a slice are relative to the slice
    par = torch.where(par >= 0, par + off, par)
    load = torch.where(load >= 0, load + off, load)
    for x, y in zip((so, par, act, load), full):
        assert same(x, y)
    assert (full[1] != torch.arange(B, device="cuda", dtype=torch.int32)).any()
