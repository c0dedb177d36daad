"""GPU: branching envs (csrc/ge_state.cu) -- per-env state records (save_states / load_states), instance replication
(gather_instances) and copy.deepcopy of the gym env, in every kernel family: round trips, forks checked against the C
oracle, `what` bits and skipped envs, slice / CUDA-graph / PDL scheduling, and a record buffer past 2^31 bytes."""
import copy
import ctypes as C
import random

import numpy as np
import pytest
import torch

import cuda_util as cu
import golden_util as gu
import graphenvs_b200 as ge
from graphenvs_b200 import BatchedGraphEnv, _native
from graphenvs_b200.batch import STATE_ALL, STATE_CLOCK, STATE_DYNAMIC, EnvStates, SliceStreams
from graphenvs_b200.instances import generate_instance
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

FAMILIES = [
    ("LongestPath-v0", 50, 200, {"parenting": 2}, False),                       # lane (cfg2 shape)
    ("ShortestPath-v0", 10, 20, {}, False),                                     # lane
    ("MaxIndependentSet-v0", 50, 200, {}, False),                               # lane
    ("PerishableProductDelivery-v0", 40, 100, {"n_products": 3, "parenting": 1}, False),   # lane
    ("ShortestPath-v0", 300, 700, {}, False),                                   # group
    ("TSP-v0", 200, 600, {"parenting": 2}, False),                              # group
    ("SteinerTree-v0", 100, 500, {"n_dests": 99}, False),                       # incremental (cfg3 shape)
    ("MulticastRouting-v0", 120, 600, {"parenting": 4, "n_dests": 5}, False),   # incremental, bestkey
    ("MulticastRouting-v0", 60, 200, {"parenting": 2, "n_dests": 3}, False),    # incremental, rev / esrc
    ("MaxIndependentSet-v0", 200, 600, {}, False),                              # incremental
    ("DistributionCenter-v0", 120, 500, {"parenting": 2}, False),               # dc, with dc_rows
    ("LongestPath-v0", 50, 200, {"parenting": 2}, True),                        # general (force_warp)
]
IDS = ["%s-N%d%s%s" % (c[0][:-3], c[1], "".join("-%s%s" % (k[0], v) for k, v in c[3].items()), "-warp" if c[4] else "")
       for c in FAMILIES]
STATE = ("head", "node_bits", "node_bits2", "edge_bits", "dist32", "bestkey", "cost", "counters", "done", "mask_bits", "mask_cnt",
         "acc", "traj")
STATIC = ("row_ptr", "col", "w32", "w64", "adj_bits", "rev", "esrc", "wsort", "wcode", "dfa", "dc_edges", "dc_rows", "wmin", "wmat",
          "src", "dest", "target_bits", "node_cost", "node_xy", "max_dist32", "targets", "in_range", "heuristic",
          "heuristic_alt", "features", "mask0_bits")
M64 = (1 << 64) - 1


def seeded_instances(env_id, params, n, base):
    inst = []
    for b in range(n):
        random.seed(base + b)
        np.random.seed(base + b)
        inst.append(generate_instance(env_id, params))
    return inst


def make_batch(cfg, B, base, **extra):
    """A loaded batch of B seeded host instances (auto-reset on); Multicast's max_distance is written back to the instances."""
    env_id, N, E, kw, warp = cfg
    env = BatchedGraphEnv(env_id, B, N, E, auto_reset=True, force_warp=warp, **kw, **extra)
    inst = seeded_instances(env_id, env.params, B, base)
    env.load_instances(inst)
    if env_id == "MulticastRouting-v0":
        md = env.t["max_dist32"].cpu().numpy()
        for b, i in enumerate(inst):
            i.max_distance = float(md[b])
    return env, inst


def snap(env):
    s = {k: env.t[k].clone() for k in STATE if k in env.t}
    if env.env_steps is not None:
        s["env_steps"] = env.env_steps.clone()
    if "mask_bytes" in env.t:
        s["mask"] = env.mask.clone()
    return s


def bits(t):
    """Bit patterns of a tensor (NaN solution costs compare equal to themselves)."""
    return t.view(torch.int64) if t.dtype == torch.float64 else t.view(torch.int32) if t.dtype == torch.float32 else t


def same(x, y):
    return torch.equal(bits(x), bits(y))


def assert_same(a, b, what=""):
    assert a.keys() == b.keys()
    for k in a:
        assert same(a[k], b[k]), "%s %s" % (what, k)


def unpack(words, A):
    return np.unpackbits(np.ascontiguousarray(words).view(np.uint8), bitorder="little")[:A].astype(bool)


# ------------------------------------------------------------------ 1. round trip
@pytest.mark.parametrize("cfg", FAMILIES, ids=IDS)
def test_round_trip_restores_state_and_replays(cfg):
    env, _ = make_batch(cfg, 150, 3000)
    env.enable_env_clock()
    env.reset()
    seed, T1, T2 = 21, 30, 20
    for t in range(T1):
        env.step_sampled(seed, t)
    at_save = snap(env)
    st = env.save_states()
    assert st.data.shape == (150, env.record_bytes()) and len(st) == 150

    def run():
        log = []
        for t in range(T1, T1 + T2):
            a = env.step_sampled(seed, t)
            log.append((a.clone(), env.reward.clone(), env.flags.clone(), env.solution_cost.clone(), env.t["mask_bits"].clone(),
                        env.t["traj"].clone()))
        torch.cuda.synchronize()
        return log
    first = run()
    env.load_states(st)
    assert_same(snap(env), at_save, "after load")
    for s0, s1 in zip(first, run()):
        for x, y in zip(s0, s1):
            assert same(x, y)


# ------------------------------------------------------------------ 2. replicate and fork against the oracle
def _traj(cs, a, o):
    cs = ((cs << 7) | (cs >> 57)) & M64
    return cs ^ (a & 0xFFFFFFFF) ^ (int(o["done"]) << 40) ^ ((o["solved"] & 3) << 44) ^ (o["status"] << 48)


def _oracle_step(oe, a, masks, j):
    o = oe.step(int(a))
    if o["done"]:
        oe.reset_state()
        masks[j] = oe.mask(reset_patch=True)
    elif o["has_mask"]:
        masks[j] = o["mask"]
    return o


@pytest.mark.parametrize("cfg", FAMILIES, ids=IDS)
def test_gather_and_fork_match_the_oracle(cfg):
    env_id = cfg[0]
    n, K = 40, 3
    src, inst = make_batch(cfg, n, 5000, structural_features=True)
    src.reset()                                                     # mask0_bits (auto-reset) is written by reset
    rng = np.random.default_rng(cfg[1])
    owner = rng.permutation(np.repeat(np.arange(n), K))             # wide env j holds src instance owner[j]
    wide = src.like(n * K)
    wide.gather_instances(src, torch.from_numpy(owner).cuda())
    ref = src.like(n * K)
    ref.load_instances([copy.deepcopy(inst[o]) for o in owner])
    ref.reset()
    statics = [k for k in STATIC if k in ref.t]
    assert statics == [k for k in STATIC if k in wide.t]
    for k in statics:
        assert same(wide.t[k], ref.t[k]), "static array %s" % k
    wide.reset()
    assert_same(snap(wide), snap(ref), "reset")

    # prefixes: every env steps P steps, with saves after 0, 3 and 7 of them
    B, seed, seed2, cps, P, T = n * K, 3, 4, (0, 3, 7), 8, 15
    saves, acts_log = {}, []
    for t in range(P):
        if t in cps:
            saves[t] = wide.save_states()
        acts_log.append(wide.sample_actions(seed, t).clone())
        wide.step_async(wide.actions_dev)
    acts_log = torch.stack(acts_log).cpu().numpy()
    records = EnvStates(torch.cat([saves[c].data for c in cps]), saves[0].signature)
    group = [np.flatnonzero(owner == owner[j]) for j in range(B)]
    cp = rng.integers(len(cps), size=B)                              # each env forks at its own prefix length ...
    parent = np.array([rng.choice(group[j]) for j in range(B)])      # ... from a random env of its instance group
    wide.load_states(records, torch.from_numpy(cp * B + parent).cuda())

    # oracle: the parent's prefix, then the forked env's own steps
    oenvs, masks, cs = [], [], [0] * B
    for j in range(B):
        oe = cu.oracle_from_instance(env_id, inst[owner[j]], src.params, features=wide.t["features"][j].cpu().numpy())
        masks.append(oe.mask(reset_patch=True))
        for t in range(cps[cp[j]]):
            a = int(acts_log[t, parent[j]])
            assert a == orc.sample_action(masks[j], seed, int(parent[j]), t)
            cs[j] = _traj(cs[j], a, _oracle_step(oe, a, masks, j))
        oenvs.append(oe)
    got = wide.t["traj"].cpu().numpy().view(np.uint64)
    assert [int(x) for x in got] == cs, "traj right after the fork"
    own = []
    for t in range(P, P + T):
        acts = wide.sample_actions(seed2, t).cpu().numpy()
        own.append(acts)
        reward, done, info = wide.step(wide.actions_dev)
        torch.cuda.synchronize()
        reward, done = reward.cpu().numpy(), done.cpu().numpy()
        solved, status = info["solved"].cpu().numpy(), info["status"].cpu().numpy()
        cost, gmask = info["solution_cost"].cpu().numpy(), wide.t["mask_bits"].cpu().numpy()
        for j, oe in enumerate(oenvs):
            tag = "%s env %d step %d" % (env_id, j, t)
            assert acts[j] == orc.sample_action(masks[j], seed2, j, t), "sampler parity " + tag
            o = _oracle_step(oe, acts[j], masks, j)
            cs[j] = _traj(cs[j], int(acts[j]), o)
            assert status[j] == o["status"] == 0, tag
            assert bool(done[j]) == o["done"] and int(solved[j]) == o["solved"], tag
            assert abs(reward[j] - o["reward"]) <= 1e-5 * max(1.0, abs(o["reward"])), tag
            if np.isnan(o["solution_cost"]):
                assert np.isnan(cost[j]), tag
            else:
                assert abs(cost[j] - o["solution_cost"]) <= 1e-5 * max(1.0, abs(o["solution_cost"])), tag
            np.testing.assert_array_equal(unpack(gmask[j], wide.desc.A), masks[j], err_msg="mask " + tag)
    obs = wide.obs_flat().cpu().numpy()
    for j, oe in enumerate(oenvs):
        np.testing.assert_allclose(obs[j], oe.obs(), rtol=1e-6, atol=0, err_msg="obs env %d" % j)
    assert [int(x) for x in wide.t["traj"].cpu().numpy().view(np.uint64)] == cs

    # an unforked batch running the concatenated actions ends with the same checksums and statistics
    own = np.stack(own)
    for c, L in enumerate(cps):
        sel = np.flatnonzero(cp == c)
        if sel.size == 0:
            continue
        plain = src.like(B)
        plain.gather_instances(src, torch.from_numpy(owner).cuda())
        plain.reset()
        for t in range(L):
            plain.step(torch.from_numpy(acts_log[t, parent]).cuda())
        for t in range(T):
            plain.step(torch.from_numpy(own[t]).cuda())
        s = torch.from_numpy(sel).cuda()
        assert same(plain.t["traj"][s], wide.t["traj"][s]), "traj, fork point %d" % L
        assert same(plain.t["acc"][:, s], wide.t["acc"][:, s]), "acc, fork point %d" % L


# ------------------------------------------------------------------ 3. what bits and skipped envs
WHAT_CFGS = [FAMILIES[0], FAMILIES[7]]


@pytest.mark.parametrize("cfg", WHAT_CFGS, ids=[IDS[0], IDS[7]])
def test_what_bits_and_out_of_range_indices(cfg):
    env, _ = make_batch(cfg, 200, 7000)
    clock = env.enable_env_clock()
    env.reset()
    for t in range(6):
        env.step_sampled(5, t)
    drawn = env.sample_actions(9, 0).clone()
    at_save = snap(env)
    st = env.save_states()
    for t in range(6, 12):
        env.step_sampled(5, t)
    later = snap(env)
    env.load_states(st, what=STATE_DYNAMIC)
    now = snap(env)
    for k in now:
        exp = later if k in ("env_steps", "acc", "traj") else at_save
        assert same(now[k], exp[k]), "DYNAMIC-only load: %s" % k
    assert not same(env.sample_actions(9, 0), drawn), "the clock was not restored, so the draws move on"
    env.load_states(st, what=STATE_DYNAMIC | STATE_CLOCK)
    assert same(clock, at_save["env_steps"]) and same(env.t["traj"], later["traj"])
    assert same(env.sample_actions(9, 0), drawn), "CLOCK restores what sample_actions draws"

    # -1 and n_records leave envs byte for byte as they were, every array of env.t included
    for t in range(12, 15):
        env.step_sampled(5, t)
    mask_before = env.mask.clone()      # (refreshes the byte view of the incremental-mask kinds first)
    before = {k: v.clone() for k, v in env.t.items()}
    before_clock = clock.clone()
    n = 50
    part = env.save_states(torch.arange(100, 150, dtype=torch.int32, device="cuda"))
    idx = torch.from_numpy(np.random.default_rng(1).integers(0, n, size=env.B)).int()
    idx[::3] = -1
    idx[1::7] = n
    env.load_states(part, idx.cuda())
    keep = (idx < 0) | (idx >= n)
    k_ = torch.nonzero(keep).flatten().cuda()
    for name, v in env.t.items():
        if name in ("acc",):
            assert same(v[:, k_], before[name][:, k_]), name
        elif v.dim() >= 1 and v.shape[0] == env.B and name in STATE + ("mask_bytes",):
            assert same(v[k_], before[name][k_]), name
        elif name not in STATE + ("mask_bytes",):
            assert same(v, before[name]), "static array %s changed" % name
    assert same(clock[k_], before_clock[k_])
    loaded = torch.nonzero(~keep).flatten().cuda()
    src_env = (idx[~keep] + 100).long().cuda()
    for name in ("head", "mask_bits", "traj", "cost"):
        if name in env.t:
            assert same(env.t[name][loaded], before[name][src_env]), name
    assert same(env.mask[loaded], mask_before[src_env])


# ------------------------------------------------------------------ 4. scheduling
def _sched_env(**kw):
    e = BatchedGraphEnv("LongestPath-v0", 1000, 50, 200, parenting=2, auto_reset=True, **kw)
    e.generate(seed=17)
    e.enable_env_clock()
    e.reset()
    for t in range(5):
        e.step_sampled(3, t)
    return e


def test_slice_descriptors_equal_the_full_batch():
    full, sliced = _sched_env(), _sched_env()
    perm = torch.randperm(1000, generator=torch.Generator().manual_seed(0)).int().cuda()
    ref = full.save_states(perm)
    rec = torch.zeros_like(ref.data)
    ss = SliceStreams(sliced, 3)
    L = sliced.lib
    ss.fork()
    for (lo, n), d, s in zip(ss.bounds, ss.descs, ss.streams):
        _native.check(L.ge_state_save(C.byref(sliced.desc), C.c_void_p(perm[lo:].data_ptr()), n, C.c_void_p(rec[lo:].data_ptr()),
                                      C.c_void_p(s.cuda_stream)))
    ss.join()
    torch.cuda.synchronize()
    assert same(rec, ref.data), "records saved per slice"
    # save through the slice descriptors themselves (env indices relative to the slice)
    rec2 = torch.zeros_like(ref.data)
    ss.fork()
    for (lo, n), d, s in zip(ss.bounds, ss.descs, ss.streams):
        _native.check(L.ge_state_save(C.byref(d), None, n, C.c_void_p(rec2[lo:].data_ptr()), C.c_void_p(s.cuda_stream)))
    ss.join()
    torch.cuda.synchronize()
    assert same(rec2, full.save_states().data)
    # load through the slice descriptors: env b <- the record of env perm[perm[b]]
    back = perm
    full.load_states(ref, back)
    ss.fork()
    for (lo, n), d, s in zip(ss.bounds, ss.descs, ss.streams):
        _native.check(L.ge_state_load(C.byref(d), C.c_void_p(rec.data_ptr()), 1000, C.c_void_p(back[lo:].data_ptr()), STATE_ALL,
                                      C.c_void_p(s.cuda_stream)))
    ss.join()
    torch.cuda.synchronize()
    assert_same(snap(full), snap(sliced), "slice load")


def test_graph_replay_and_pdl_equal_eager():
    K = 12
    perm = torch.randperm(1000, generator=torch.Generator().manual_seed(1)).int().cuda()
    runs = {}
    for mode in ("eager", "graph", "pdl"):
        e = _sched_env()
        if mode == "pdl":
            e.enable_pdl()
        buf = e.save_states()
        log = []

        def body():
            e.step_sampled(7, 0)
            e.save_states(out=buf)
            e.load_states(buf, perm)
            e.step_sampled(7, 1)
        if mode == "graph":
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                body()
            for _ in range(K):
                g.replay()
                log.append(snap(e))
        else:
            for _ in range(K):
                body()
                log.append(snap(e))
        torch.cuda.synchronize()
        runs[mode] = log
    for mode in ("graph", "pdl"):
        for i, (a, b) in enumerate(zip(runs["eager"], runs[mode])):
            assert_same(a, b, "%s replay %d" % (mode, i))


# ------------------------------------------------------------------ 5. scale: a record buffer past 2^31 bytes
def test_cfg5_multicast_records_past_2gb():
    # 262,144 cfg5 Multicast envs fill exactly 2^31 bytes of 8,192-byte records; 32 more put the last ones past it
    B, N, E, T, seed = 262144 + 32, 500, 4000, 12, 4242
    env = BatchedGraphEnv("MulticastRouting-v0", B, N, E, n_dests=3, parenting=4, auto_reset=True)
    env.generate(seed=6)
    env.reset()
    for t in range(T):
        env.sample_actions(seed, t)
        env.step_async(env.actions_dev)
    st = env.save_states()
    assert (B - 1) * st.data.shape[1] > 2 ** 31, st.data.shape
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(5))
    check = np.concatenate([np.arange(0, 86), np.arange(B // 2 - 43, B // 2 + 42), np.arange(B - 85, B)])
    srcs = perm[check].numpy()
    pick = torch.from_numpy(srcs).long().cuda()
    expect = {k: env.t[k][pick].clone() for k in STATE if k in env.t and k != "acc"}
    expect_acc = env.t["acc"][:, pick].clone()
    env.load_states(st, perm.int().cuda())
    del st
    rows = torch.from_numpy(check).long().cuda()
    for k, v in expect.items():
        assert same(env.t[k][rows], v), k
    assert same(env.t["acc"][:, rows], expect_acc)
    # the loaded envs carry the state the oracle reaches on the envs their records came from
    traj = env.t["traj"][rows].cpu().numpy().view(np.uint64)
    acc = env.t["acc"][:, rows].cpu().numpy()
    gmask = env.t["mask_bits"][rows].cpu().numpy()
    for i, s in enumerate(srcs):
        ins = env.export_instances(int(s), 1)[0]
        oe = cu.oracle_from_instance("MulticastRouting-v0", ins, env.params)
        sr, ep, cs = orc.rollout([oe], T, seed, env_id0=int(s))
        assert traj[i] == cs[0] and int(acc[0, i]) == ep[0], "env %d (record of env %d)" % (check[i], s)
        assert abs(acc[2, i] - sr[0]) <= 1e-4 + 1e-5 * abs(sr[0])
        np.testing.assert_array_equal(unpack(gmask[i], 2 * E), oe.mask(reset_patch=False))


# ------------------------------------------------------------------ 6. copy.deepcopy of the gym env
_seen, DEEP = set(), []
for _m, _r in gu.all_cases():
    if _m["env_id"] not in _seen and _m["N"] <= 50:
        _seen.add(_m["env_id"])
        DEEP.append(_m)


def _same_info(a, b):
    assert a.keys() == b.keys()
    for k in a:
        x, y = a[k], b[k]
        if isinstance(x, np.ndarray):
            np.testing.assert_array_equal(x, y)
        elif isinstance(x, float) and np.isnan(x):
            assert np.isnan(y)
        else:
            assert x == y, k


@pytest.mark.parametrize("m", DEEP, ids=[m["env_id"][:-3] for m in DEEP])
def test_deepcopy_branches_the_gym_env(m):
    assert len(DEEP) == 9
    env = ge.make(m["env_id"], **m["kwargs"])
    rng = np.random.default_rng(0)
    for sd in range(m["seed"], m["seed"] + 20):          # mid-episode: an instance whose episode outlasts two steps
        obs, info = env.reset(seed=sd)
        mask, done = info["mask"], False
        for _ in range(2):
            obs, r, done, _, info = env.step(int(rng.choice(np.flatnonzero(mask))))
            mask = info.get("mask", mask)
            if done:
                break
        if not done:
            break
    assert not done
    twin = copy.deepcopy(env)
    assert twin.core is not env.core and twin.instance is not env.instance
    np.testing.assert_array_equal(twin._obs(), env._obs())
    for _ in range(40):
        a = int(rng.choice(np.flatnonzero(mask)))
        keep = env._obs()
        o2, r2, d2, t2, i2 = twin.step(a)
        np.testing.assert_array_equal(env._obs(), keep)   # stepping the copy leaves the original as it was
        o1, r1, d1, t1, i1 = env.step(a)
        np.testing.assert_array_equal(o1, o2)
        assert (r1, d1, t1) == (r2, d2, t2)
        _same_info(i1, i2)
        if d1:
            break
        mask = i1.get("mask", mask)
