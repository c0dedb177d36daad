"""GPU: stochastic beam search (ge_beam_expand_sampled, graphenvs_b200.StochasticBeamSearch).  The expand kernel against a
float64 restatement (log-probs, node keys and the bookkeeping exact, keys within a stated tolerance); width nesting; width 1
against ancestral sampling; exhaustive search on tiny instances against the C oracle's enumeration; the sampling distribution,
the inclusion probabilities and the priority-sampling estimator on a tiny instance; every family at W = 8 against the oracle;
and CUDA-graph / PDL / slice / rank-slice scheduling.  Every test uses fixed seeds: nothing here can flake."""
import ctypes as C
import itertools
import random

import numpy as np
import pytest
import torch
from scipy import stats

import cuda_util as cu
import graphenvs_b200 as ge
from graphenvs_b200 import BatchedGraphEnv, _native, policy as pol
from graphenvs_b200.instances import generate_instance
from test_cuda_beam import TINY, _close, _dummy_desc, enumerate_trajectories, replay_scores, same, table_policy, trim
from test_cuda_env_state import FAMILIES, IDS, make_batch

pytestmark = pytest.mark.gpu

NEG = float("-inf")
M64 = (1 << 64) - 1


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


# ------------------------------------------------------------------ the documented formulas, restated in numpy
def mix32(seed, env, t):
    """csrc/ge_common.cuh:mix32 in numpy uint64 arithmetic (wrapping); every argument broadcasts."""
    with np.errstate(over="ignore"):
        seed, env, t = (np.asarray(x, dtype=np.uint64) for x in (seed, env, t))
        z = seed + np.uint64(0x9E3779B97F4A7C15) * (env * np.uint64(0x100000001) + ((t << np.uint64(32)) | np.uint64(0x5bd1e995)))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
        return z >> np.uint64(32)


def gumbel64(node_key, a):
    """g = -log(-log(u)) in float64 of the kernel's u: fl32((h >> 8) + 0.5) / 2^24 (the sum rounds to even once h >> 8 >= 2^23,
    which moves the largest g by up to a quarter), at most 1 - 2^-24; h = mix32(node_key, a, 0x85EBCA6B)."""
    h = mix32(node_key, a, 0x85EBCA6B)
    u = ((h >> np.uint64(8)).astype(np.float32) + np.float32(0.5)).astype(np.float64) / 2.0 ** 24
    return -np.log(-np.log(np.minimum(u, 1 - 2.0 ** -24)))


def child_key(h, a):
    """(uint64) mix32(h, a, 0x2545F491) << 32 | mix32(h ^ 0x9E3779B97F4A7C15, a, 0x6C8E9CF5)."""
    h = np.asarray(h, dtype=np.uint64)
    return (mix32(h, a, 0x2545F491) << np.uint64(32)) | mix32(h ^ np.uint64(0x9E3779B97F4A7C15), a, 0x6C8E9CF5)


def root_key(seed, i):
    """(uint64) mix32(seed, i, 0x52DCE729) << 32 | mix32(seed ^ 0xD1B54A32D192ED03, i, 0x52DCE729)."""
    return (mix32(seed, i, 0x52DCE729) << np.uint64(32)) | mix32(seed ^ 0xD1B54A32D192ED03, i, 0x52DCE729)


def log1mexp(x):
    with np.errstate(divide="ignore"):
        return np.where(x > -np.log(2), np.log(-np.expm1(np.minimum(x, 0))), np.log1p(-np.exp(np.minimum(x, -np.log(2)))))


def conditioned(T, Z, x):
    """Kool et al. 2019, appendix: the key of a child whose perturbed log-prob lies x <= 0 below its siblings' maximum Z, given
    its parent's key T: -log(e^-T - e^-Z + e^-(Z + x)), in the stable form of the header."""
    v = (T - Z - x) + log1mexp(x)
    return T - (np.maximum(v, 0) + np.log1p(np.exp(-np.abs(v))))


# ------------------------------------------------------------------ 1. the kernel against a float64 restatement
def _expand_sampled(d, W, logits, logp, key, node_key, threshold=True):
    B, dev = d.B, logits.device
    out = [torch.full((B,), 7.0, device=dev), torch.full((B,), 7.0, device=dev), torch.full((B,), 7, dtype=torch.int64, device=dev)]
    out += [torch.full((B,), 7, dtype=torch.int32, device=dev) for _ in range(3)]
    thr = torch.full((B // W,), 7.0, device=dev) if threshold else None
    _native.check(_native.lib().ge_beam_expand_sampled(C.byref(d), W, _p(logits), pol._DTYPES[logits.dtype], _p(logp), _p(key),
                                                       _p(node_key), *[_p(t) for t in out], _p(thr),
                                                       C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out + [thr]


# Tolerance of a key.  With lse taken from the native forward (as the exact checks do), the float32 kernel and the float64
# restatement differ by the rounding of g_a (two logf of the same float32 u, <= 2 ulp each), of s_a = l_a + g_a and S_b, of D_b and of the transform's
# few operations: each an error of at most 2^-23 relative to the magnitudes involved.  G is a function of (T, D, x) whose
# partial derivatives are bounded by 1, 1 and e^max(D, 0) (dG/dx = 1 / (1 - e^x (1 - e^-D))), so the key's error is at most
# ~ 8 * 2^-23 * e^max(D, 0) * (1 + |T| + |logp| + |lse| + |l_a| + |g_a| + |S_b|).  The tolerance is 2^-19 times that bracket:
# twice the bound.
def key_tolerance(D, T, logp, lse, l, g, S):
    return 2.0 ** -19 * np.exp(np.maximum(D, 0.0)) * (1 + abs(T) + abs(logp) + abs(lse) + np.abs(l) + np.abs(g) + abs(S))


def reference_sampled(logits, valid, done, logp, key, node_key, W):
    """Per group, every candidate with its float64 key G, tolerance, exact float32 log-prob and exact child node key, in the
    order (G desc, parent, action) of the float64 keys.  lse comes from ge_masked_log_prob (checked against float64 by
    test_cuda_policy), log-probs are float32 sums in torch as in test_cuda_beam.reference_expand."""
    B, A = logits.shape
    AW = (A + 31) // 32
    packed = np.packbits(np.pad(valid, ((0, 0), (0, AW * 32 - A))), axis=1, bitorder="little").view(np.int32)
    mb = torch.from_numpy(packed.copy()).cuda()
    lp, ent, lse = (torch.empty(B, device="cuda") for _ in range(3))
    acts = torch.zeros(B, dtype=torch.int32, device="cuda")
    _native.check(_native.lib().ge_masked_log_prob(_p(logits), pol._DTYPES[logits.dtype], B, A, _p(mb), _p(acts), _p(lp), _p(ent), _p(lse), None))
    phi = (torch.from_numpy(logp).cuda()[:, None] + (logits.float() - lse[:, None])).cpu().numpy()   # fl32(logp + fl32(l - lse))
    lse = lse.cpu().numpy().astype(np.float64)
    l64 = logits.float().cpu().numpy().astype(np.float64)
    groups = []
    for g in range(B // W):
        cand = []                                              # (G, tol, parent, action, phi, node key)
        for b in range(g * W, g * W + W):
            T = float(key[b])
            if T == NEG:
                continue
            if done[b]:
                cand.append((T, 0.0, b, -1, logp[b], int(node_key[b])))
                continue
            av = np.flatnonzero(valid[b])
            if av.size == 0:
                continue
            gum = gumbel64(node_key[b], av)
            s = l64[b, av] + gum
            S = s.max()
            Z = float(logp[b]) + (S - lse[b])
            G = conditioned(T, Z, s - S)
            tol = key_tolerance(T - Z, T, float(logp[b]), lse[b], l64[b, av], gum, S)
            ck = child_key(node_key[b], av)
            cand.extend(zip(G.tolist(), tol.tolist(), [b] * av.size, av.tolist(), phi[b, av].tolist(), ck.tolist()))
        cand.sort(key=lambda c: (-c[0], c[2], c[3]))
        groups.append(cand)
    return groups


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("A", [7, 50, 200, 8000])
@pytest.mark.parametrize("W", [1, 2, 5, 16, 32])
def test_expand_sampled_against_reference(W, A, dtype):
    rng = np.random.default_rng(W * 100019 + A + (dtype == torch.bfloat16))
    G = max(2, 160 // W)
    B = G * W
    vals = (rng.standard_normal((B, A)) * 2).astype(np.float32)       # continuous logits
    density = rng.choice([0.0, 0.03, 0.3, 1.0], size=B)
    valid = rng.random((B, A)) < density[:, None]
    done = rng.random(B) < 0.2
    logp = (-rng.random(B) * 6).astype(np.float32)
    key = (logp + rng.gumbel(size=B)).astype(np.float32)               # T = logp + Gumbel(0): the keys a search carries
    key[rng.random(B) < 0.2] = NEG
    root = rng.random(B // W) < 0.5                                    # some groups hold one root and dead slots
    for g in np.flatnonzero(root):
        logp[g * W], key[g * W] = 0.0, rng.gumbel()
        key[g * W + 1:g * W + W] = NEG
    node_key = rng.integers(0, M64, size=B, dtype=np.uint64, endpoint=True)
    vals[~valid] = np.nan                                              # invalid logits are never read
    logits = torch.from_numpy(vals).cuda().to(dtype)
    AW = (A + 31) // 32
    packed = np.packbits(np.pad(valid, ((0, 0), (0, AW * 32 - A))), axis=1, bitorder="little").view(np.uint32).copy()
    if A % 32:
        packed[:, -1] |= np.uint32(0xFFFFFFFF) << np.uint32(A % 32)   # stray bits past A are ignored
    mask = torch.from_numpy(packed.view(np.int32)).cuda()
    done_t = torch.from_numpy(done.astype(np.uint8)).cuda()
    d = _dummy_desc(B, A, mask, done_t)
    ref = reference_sampled(logits, valid, done, logp, key, node_key, W)
    ins = [torch.from_numpy(logp).cuda(), torch.from_numpy(key).cuda(), torch.from_numpy(node_key.view(np.int64)).cuda()]
    out = _expand_sampled(d, W, logits, *ins)
    torch.cuda.synchronize()
    lo, ko, nko, par, act, load, thr = (t.cpu().numpy() for t in out)
    nko = nko.view(np.uint64)
    exemptions, checked = 0, 0
    for g, cand in enumerate(ref):
        idx = {(c[2], c[3]): c for c in cand}
        n = min(W, len(cand))
        for j in range(W):
            b = g * W + j
            if j >= n:                                                 # empty slots
                assert (par[b], act[b], load[b], nko[b]) == (-1, -1, -1, 0) and lo[b] == NEG and ko[b] == NEG, (g, j)
                continue
            p, a = int(par[b]), int(act[b])
            assert (p, a) in idx, (g, j, p, a)
            c = idx[(p, a)]
            assert load[b] == (-1 if p == b else p)
            assert np.float32(lo[b]).view(np.int32) == np.float32(c[4]).view(np.int32), (g, j)    # log-prob: bit for bit
            assert int(nko[b]) == c[5], (g, j)                                                       # node key: exact
            if a < 0 or c[0] == float(key[p]):                         # a stay, or the best child: T inherited exactly
                assert ko[b] == np.float32(key[p]), (g, j)
            assert abs(float(ko[b]) - c[0]) <= c[1], (g, j, float(ko[b]), c[0], c[1])
            checked += 1
            r = cand[j]                                                # the reference's candidate for this slot
            if (r[2], r[3]) != (p, a):
                assert abs(r[0] - c[0]) <= r[1] + c[1], "slot %d of group %d: selection differs beyond the tolerance" % (j, g)
                exemptions += 1
            if j + 1 < n:                                              # the output follows the total order
                b2 = b + 1
                assert ko[b] > ko[b2] or (ko[b] == ko[b2] and (par[b], act[b]) < (par[b2], act[b2])), (g, j)
        if len(cand) > W:
            assert abs(float(thr[g]) - cand[W][0]) <= cand[W][1] + max(c[1] for c in cand[:W + 1]), g
            assert thr[g] <= ko[g * W + W - 1]
        else:
            assert thr[g] == NEG, g
    assert checked > 0
    assert exemptions == 0, "%d selections within the tolerance of a tie (continuous logits: expected none)" % exemptions
    # deterministic, and threshold = NULL changes nothing else
    again = _expand_sampled(d, W, logits, *ins)
    assert all(same(x, y) for x, y in zip(again, out))
    no_thr = _expand_sampled(d, W, logits, *ins, threshold=False)
    assert all(same(x, y) for x, y in zip(no_thr[:-1], out[:-1]))


# ------------------------------------------------------------------ decoding helpers
def decode(venv, W, policy, seed, **kw):
    return ge.StochasticBeamSearch(venv, width=W, seed=seed).run(policy, **kw)


def pad(x, T):
    """[..., t] int32 actions padded with -1 to T steps."""
    if x.shape[-1] >= T:
        return x
    return torch.cat([x, torch.full(x.shape[:-1] + (T - x.shape[-1],), -1, dtype=x.dtype, device=x.device)], dim=-1)


# ------------------------------------------------------------------ 2. width nesting
@pytest.mark.parametrize("cfg", FAMILIES, ids=IDS)
def test_width_nesting(cfg):
    venv, _ = make_batch(cfg, 48, 21000)
    pol_fn = table_policy(venv, 1, scale=1.5, seed=13)
    small, large = decode(venv, 4, pol_fn, 77), decode(venv, 8, pol_fn, 77)
    T = max(small.beams.actions.shape[-1], large.beams.actions.shape[-1])
    a4, a8 = pad(small.beams.actions, T), pad(large.beams.actions, T)[:, :4]
    assert torch.equal(a4, a8)
    assert same(small.beams.log_prob, large.beams.log_prob[:, :4].contiguous())
    assert same(small.beams.key, large.beams.key[:, :4].contiguous())
    assert same(small.kappa, large.beams.key[:, 4].contiguous())
    assert bool((small.beams.key[:, 0] > NEG).all())


# ------------------------------------------------------------------ 3. width 1 is ancestral sampling
def ancestral(venv, policy, seed, max_steps):
    """Per instance: from the root key, take argmax over valid a of fl32(l_a + g_a) (g_a rounded to float32, lowest action on
    ties), step, and chain node keys with child_key."""
    ref = venv.like(venv.B, auto_reset=False)
    ref.gather_instances(venv)
    ref.reset()
    ref.t["acc"].zero_()
    G, A = venv.B, venv.desc.A
    nk = root_key(seed, np.arange(G, dtype=np.uint64) + np.uint64(venv.desc.env_id0))
    seqs = [[] for _ in range(G)]
    acts_all = np.arange(A, dtype=np.uint64)
    for t in range(max_steps):
        done = ref.t["done"].cpu().numpy().astype(bool)
        if done.all():
            break
        logits = policy(ref).float().cpu().numpy()
        mb = ref.t["mask_bits"].cpu().numpy().view(np.uint8)
        valid = np.unpackbits(mb, axis=1, bitorder="little")[:, :A].astype(bool)
        g32 = gumbel64(nk[:, None], acts_all[None, :]).astype(np.float32)
        s = np.where(valid, logits + g32, -np.inf).astype(np.float32)
        a = np.where(done | ~valid.any(1), -1, s.argmax(1)).astype(np.int32)
        for b in np.flatnonzero(a >= 0):
            seqs[b].append(int(a[b]))
        nk = np.where(a >= 0, child_key(nk, np.maximum(a, 0).astype(np.uint64)), nk)
        ref.step(torch.from_numpy(a).cuda())
    return seqs


@pytest.mark.parametrize("cfg", FAMILIES, ids=IDS)
def test_width_one_is_ancestral_sampling(cfg):
    venv, _ = make_batch(cfg, 40, 9100)
    pol_fn = table_policy(venv, 1, scale=2.0, seed=3)
    res = decode(venv, 1, pol_fn, 2024)
    seqs = ancestral(venv, pol_fn, 2024, res.steps)
    for g in range(venv.B):
        assert trim(res.beams.actions[g, 0].cpu().numpy()) == seqs[g], "instance %d" % g
    s, _ = replay_scores(venv, 1, pol_fn, res.beams.actions)
    assert same(s, res.beams.log_prob.flatten())


# ------------------------------------------------------------------ 4. exhaustive on tiny instances
def tiny_instances(env_id, N, E, kw, W, count, lo=1):
    probe = BatchedGraphEnv(env_id, 1, N, E, **kw)
    inst, trees = [], []
    for s in range(300):
        random.seed(s)
        np.random.seed(s)
        ins = generate_instance(env_id, probe.params)
        tree = enumerate_trajectories(cu.oracle_from_instance(env_id, ins, probe.params), W)
        if tree is not None and len(tree) >= lo:
            inst.append(ins)
            trees.append(tree)
        if len(inst) == count:
            break
    assert len(inst) == count
    return inst, trees


@pytest.mark.parametrize("tiny", TINY, ids=[t[0][:-3] for t in TINY])
def test_exhaustive_on_tiny_instances(tiny):
    env_id, N, E, kw = tiny
    W = 32
    inst, trees = tiny_instances(env_id, N, E, kw, W, 6)
    venv = BatchedGraphEnv(env_id, len(inst), N, E, **kw)
    venv.load_instances(inst)
    res = decode(venv, W, table_policy(venv, 1, scale=1.0, seed=5), 9)
    assert bool((res.kappa == NEG).all())
    for g, tree in enumerate(trees):
        alive = (res.beams.key[g] > NEG).cpu().numpy()
        done = res.beams.done[g].cpu().numpy()
        got = {}
        for j in np.flatnonzero(alive):
            assert done[j], "instance %d slot %d did not finish" % (g, j)
            q = tuple(trim(res.beams.actions[g, j].cpu().numpy()))
            assert q not in got, "instance %d: %s twice" % (g, q)
            got[q] = j
        assert set(got) == set(tree), "instance %d" % g
        for q, j in got.items():
            ret, o = tree[q]
            assert _close(res.beams.ret[g, j].item(), ret), (g, q)
            sol = 0.0 if np.isnan(o["solution_cost"]) else o["solution_cost"]
            assert _close(res.beams.solution_cost[g, j].item(), sol), (g, q)
            assert bool(res.beams.solved[g, j]) == (o["solved"] == 1), (g, q)
        w = res.beams.weight[g][torch.from_numpy(alive).cuda()]
        lp = res.beams.log_prob[g][torch.from_numpy(alive).cuda()].double()
        assert torch.equal(w, torch.exp(lp))
        assert abs(w.sum().item() - 1.0) <= 1e-5, g
        assert bool((res.beams.weight[g][torch.from_numpy(~alive).cuda()] == 0).all())


# ------------------------------------------------------------------ 5. the distribution
DIST_SEED, DIST_GROUPS, DIST_K, DIST_SIGMAS = 31337, 32768, 3, 5.0


def test_sampling_distribution_inclusion_and_estimator():
    """One ShortestPath instance with 6-12 trajectories, replicated to 32,768 groups (each its own noise through its instance
    id), K = 3, seed 31337.  Slot 0 is a draw from p(y); slot membership matches the without-replacement inclusion
    probabilities; the priority-sampling estimate of E[f] is unbiased.  Margins: 5 standard errors, chi-square p > 1e-6."""
    env_id, N, E, kw = TINY[0]
    inst, trees = tiny_instances(env_id, N, E, kw, 12, 1, lo=6)
    tree = trees[0]
    Gn, K = DIST_GROUPS, DIST_K
    one = BatchedGraphEnv(env_id, 1, N, E, **kw)
    one.load_instances(inst)
    venv = BatchedGraphEnv(env_id, Gn, N, E, **kw)
    venv.gather_instances(one, torch.zeros(Gn, dtype=torch.int32, device="cuda"))
    gen = torch.Generator(device="cuda").manual_seed(17)
    tab = torch.randn((N, venv.desc.A), generator=gen, device="cuda") * 1.5

    def policy(env):
        return tab[env.t["head"].long().clamp(0, N - 1)]

    res = decode(venv, K, policy, DIST_SEED)
    ys = sorted(tree)
    # exact p(y) by replay of every trajectory
    T = max(len(y) for y in ys)
    acts = torch.tensor([list(y) + [-1] * (T - len(y)) for y in ys], dtype=torch.int32, device="cuda")
    s, _ = replay_scores(one, len(ys), policy, acts.view(1, len(ys), T))
    p = np.exp(s.double().cpu().numpy())
    assert abs(p.sum() - 1.0) < 1e-5
    p /= p.sum()
    ret = np.array([tree[y][0] for y in ys])
    index = {y: i for i, y in enumerate(ys)}
    seq = res.beams.actions.cpu().numpy()
    assert bool(res.beams.done.all()) and bool((res.beams.key > NEG).all())
    sampled = np.array([[index[tuple(trim(seq[g, j]))] for j in range(K)] for g in range(Gn)])
    assert all(len(set(r)) == K for r in sampled), "sequences within a group are distinct"
    # slot 0 ~ p(y)
    counts = np.bincount(sampled[:, 0], minlength=len(ys))
    chi2 = ((counts - Gn * p) ** 2 / (Gn * p)).sum()
    assert stats.chi2.sf(chi2, len(ys) - 1) > 1e-6, (counts, Gn * p)
    # inclusion probabilities, enumerated over ordered triples
    incl = np.zeros(len(ys))
    for tr in itertools.permutations(range(len(ys)), K):
        q, rest = 1.0, 1.0
        for i in tr:
            q *= p[i] / rest
            rest -= p[i]
        incl[list(tr)] += q
    freq = np.bincount(sampled.ravel(), minlength=len(ys)) / Gn
    se = np.sqrt(incl * (1 - incl) / Gn)
    assert np.all(np.abs(freq - incl) <= DIST_SIGMAS * se), (freq, incl)
    # priority sampling: mean_g sum_y w_y f(y) estimates sum_y p(y) f(y)
    w = res.beams.weight.cpu().numpy()
    assert np.isfinite(w).all() and bool((res.kappa > NEG).all())
    for f in (ret, np.ones(len(ys))):
        est = (w * f[sampled]).sum(1)
        assert abs(est.mean() - (p * f).sum()) <= DIST_SIGMAS * est.std() / np.sqrt(Gn)


# ------------------------------------------------------------------ 6. every family at W = 8 against the oracle
@pytest.mark.parametrize("cfg", FAMILIES, ids=IDS)
def test_every_family_against_the_oracle(cfg):
    env_id = cfg[0]
    W, G = 8, 64
    venv, inst = make_batch(cfg, G, 12000)
    pol_fn = table_policy(venv, W, scale=2.0, seed=11)
    res = decode(venv, W, pol_fn, 5)
    alive = res.beams.key > NEG
    s, acc = replay_scores(venv, W, pol_fn, torch.where(alive[..., None], res.beams.actions, -1))
    a = alive.flatten()
    assert same(s[a], res.beams.log_prob.flatten()[a]), "log_prob is the sum of masked_log_prob terms"
    assert torch.equal(acc[2][a], res.beams.ret.flatten()[a])
    seq, done = res.beams.actions.cpu().numpy(), res.beams.done.cpu().numpy()
    ret, cost, solved = res.beams.ret.cpu().numpy(), res.beams.solution_cost.cpu().numpy(), res.beams.solved.cpu().numpy()
    keys = res.beams.key.cpu().numpy()
    assert done[alive.cpu().numpy()].any() or env_id == "PerishableProductDelivery-v0"
    for g in range(G):
        live = np.flatnonzero(keys[g] > NEG)
        assert np.all(np.diff(keys[g, live]) <= 0), g
        seqs = [tuple(trim(seq[g, j])) for j in live]
        assert len(set(seqs)) == len(seqs), "instance %d: repeated sequence" % g
        for j, q in zip(live, seqs):
            if not done[g, j]:
                continue
            oe = cu.oracle_from_instance(env_id, inst[g], venv.params)
            r, o = 0.0, None
            for x in q:
                assert o is None or not o["done"]
                o = oe.step(x)
                assert o["status"] == 0, (g, j, x)
                r += o["reward"]
            assert o["done"], (g, j)
            tag = "%s instance %d slot %d" % (env_id, g, j)
            assert _close(ret[g, j], r), tag
            assert _close(cost[g, j], 0.0 if np.isnan(o["solution_cost"]) else o["solution_cost"]), tag
            assert bool(solved[g, j]) == (o["solved"] == 1), tag


# ------------------------------------------------------------------ 7. scheduling
def _sched(pdl=False, **kw):
    venv = BatchedGraphEnv("LongestPath-v0", 128, 50, 200, parenting=2, auto_reset=True, **kw)
    venv.generate(seed=23)
    sbs = ge.StochasticBeamSearch(venv, width=8, seed=99)
    if pdl:
        sbs.wide.enable_pdl()
    return venv, sbs


def test_graph_replay_and_pdl_equal_eager():
    T = 12
    runs = {}
    for mode in ("eager", "graph", "pdl"):
        venv, sbs = _sched(pdl=mode == "pdl")
        pol_fn = table_policy(venv, 8, scale=0.5, seed=4)
        sbs.start()
        sbs.reserve(T)
        if mode == "graph":
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                for _ in range(T):
                    sbs.advance(pol_fn(sbs.wide))
            g.replay()
        else:
            for _ in range(T):
                sbs.advance(pol_fn(sbs.wide))
        torch.cuda.synchronize()
        runs[mode] = (sbs._parents[:T].clone(), sbs._actions[:T].clone(), sbs._thresholds[:T].clone(), sbs.score.clone(),
                      sbs.key.clone(), sbs.node_key.clone(), sbs.wide.t["acc"].clone(), sbs.wide.t["traj"].clone(),
                      sbs.wide.t["mask_bits"].clone(), sbs.wide.t["done"].clone())
    for mode in ("graph", "pdl"):
        for i, (x, y) in enumerate(zip(runs["eager"], runs[mode])):
            assert same(x, y), "%s item %d" % (mode, i)
    assert (runs["eager"][1][1:] >= 0).any() and (runs["eager"][0][1] != torch.arange(1024, device="cuda")).any()
    assert bool((runs["eager"][2] > NEG).any())


def test_expand_over_slices_equals_one_descriptor():
    venv, sbs = _sched()
    pol_fn = table_policy(venv, 8, scale=0.5, seed=5)
    sbs.start()
    for _ in range(4):
        sbs.advance(pol_fn(sbs.wide))
    wide = sbs.wide
    logits = pol_fn(wide).to(torch.bfloat16).contiguous()
    ins = (sbs.score, sbs.key, sbs.node_key)
    full = _expand_sampled(wide.desc, 8, logits, *ins)
    B, lo = wide.B, 512
    parts = _expand_sampled(wide.desc, 8, logits, *ins)        # overwritten slice by slice below
    for t in parts:
        t.fill_(7)
    for start, n in ((0, lo), (lo, B - lo)):
        d = wide.slice_desc(start, n)
        _native.check(wide.lib.ge_beam_expand_sampled(C.byref(d), 8, _p(logits[start:]), pol._DTYPES[logits.dtype],
                                                      *[_p(t[start:]) for t in ins], *[_p(t[start:]) for t in parts[:6]],
                                                      _p(parts[6][start // 8:]), wide._stream()))
    torch.cuda.synchronize()
    off = torch.zeros(B, dtype=torch.int32, device="cuda")
    off[lo:] = lo                                               # indices of a slice are relative to the slice
    parts[3] = torch.where(parts[3] >= 0, parts[3] + off, parts[3])
    parts[5] = torch.where(parts[5] >= 0, parts[5] + off, parts[5])
    for x, y in zip(parts, full):
        assert same(x, y)
    assert (full[3] != torch.arange(B, device="cuda", dtype=torch.int32)).any()


def test_rank_slice_draws_what_the_full_batch_draws():
    """Instances [40, 104) of a 128-instance batch, loaded on their own with env_id0 = 40, decode to the same sequences, keys
    and weights as in the full batch (the policy depends on the global instance id only)."""
    cfg = FAMILIES[0]
    venv, inst = make_batch(cfg, 128, 31000)
    lo, n, W = 40, 64, 8
    part, _ = make_batch(cfg, n, 31000 + lo, env_id0=lo)
    gen = torch.Generator(device="cuda").manual_seed(6)
    tab = torch.randn((128, venv.N, venv.desc.A), generator=gen, device="cuda")

    def policy_for(first):
        def policy(env):
            g = first + torch.arange(env.B, device="cuda") // W
            return tab[g, env.t["head"].long().clamp(0, venv.N - 1)]
        return policy

    full = decode(venv, W, policy_for(0), 1234)
    sub = decode(part, W, policy_for(lo), 1234)
    T = max(full.beams.actions.shape[-1], sub.beams.actions.shape[-1])
    assert torch.equal(pad(full.beams.actions, T)[lo:lo + n], pad(sub.beams.actions, T))
    for k in ("log_prob", "key", "ret"):
        assert torch.equal(getattr(full.beams, k)[lo:lo + n], getattr(sub.beams, k)), k
    assert same(full.kappa[lo:lo + n].contiguous(), sub.kappa)
    assert torch.equal(full.beams.weight[lo:lo + n].isnan(), sub.beams.weight.isnan())
    fin = ~sub.beams.weight.isnan()
    assert torch.equal(full.beams.weight[lo:lo + n][fin], sub.beams.weight[fin])
