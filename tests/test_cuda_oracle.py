"""GPU: CUDA engine vs the C oracle on seeded instances (host generator = the reference's draws),
device-sampled random valid actions, auto-reset on.  Sizes go beyond the golden fixtures
(N > 64 exercises the multi-word bitset paths, N <= 64 the register fast paths)."""
import random

import numpy as np
import pytest
import torch

import cuda_util as cu
from graphenvs_b200 import BatchedGraphEnv
from graphenvs_b200.instances import generate_instance
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

CONFIGS = [
    ("ShortestPath-v0", 10, 20, {}, 24),
    ("ShortestPath-v0", 100, 300, {}, 40),
    ("ShortestPath-v0", 300, 700, {}, 60),                    # group-per-env family, 16 lanes per env
    ("ShortestPath-v0", 600, 1500, {}, 60),                   # 32 lanes per env
    ("ShortestPath-v0", 1100, 3000, {}, 15),                  # NW = 35 > 32: general family, multi-word-per-lane sets
    ("DensestSubgraph-v0", 1100, 4000, {"parenting": 1}, 15),
    ("SteinerTree-v0", 1100, 3000, {"n_dests": 6}, 20),       # incremental kernel without register-resident bitsets
    ("MulticastRouting-v0", 1100, 3000, {"parenting": 4, "n_dests": 4}, 20),
    ("DistributionCenter-v0", 1100, 3000, {"parenting": 2, "target_count": 40}, 10),
    ("LongestPath-v0", 100, 300, {"parenting": 1}, 60),
    ("LongestPath-v0", 80, 200, {"parenting": 0}, 40),
    ("TSP-v0", 70, 300, {"parenting": 1}, 80),
    ("TSP-v0", 130, 8385, {"parenting": 1}, 140),            # complete graph
    ("TSP-v0", 300, 1200, {"parenting": 1}, 100),
    ("DensestSubgraph-v0", 300, 1500, {"parenting": 1}, 60),
    ("DensestSubgraph-v0", 600, 3000, {"parenting": 0}, 60),
    ("LongestPath-v0", 50, 200, {"parenting": 2}, 60),       # BASELINE config 2 shape
    ("LongestPath-v0", 33, 70, {"parenting": 2}, 40),
    ("LongestPath-v0", 64, 200, {"parenting": 2}, 60),
    ("LongestPath-v0", 32, 80, {"parenting": 3}, 40),
    ("LongestPath-v0", 20, 50, {"parenting": 0}, 30),
    ("TSP-v0", 64, 300, {"parenting": 2}, 80),
    ("TSP-v0", 24, 276, {"parenting": 2}, 40),
    ("MaxIndependentSet-v0", 50, 200, {}, 60),
    ("DensestSubgraph-v0", 64, 300, {"parenting": 1}, 40),
    ("DensestSubgraph-v0", 30, 100, {"parenting": 0}, 30),
    ("LongestPath-v0", 100, 260, {"parenting": 2}, 60),
    ("LongestPath-v0", 90, 200, {"parenting": 3}, 60),
    ("LongestPath-v0", 40, 100, {"parenting": 1}, 40),
    ("SteinerTree-v0", 100, 500, {"n_dests": 99}, 120),      # config 3 shape
    ("SteinerTree-v0", 60, 150, {"n_dests": 5}, 80),
    ("TSP-v0", 40, 120, {"parenting": 1}, 50),
    ("TSP-v0", 40, 120, {"parenting": 2}, 50),
    ("TSP-v0", 70, 2415, {"parenting": 2}, 80),               # complete graph, N > 64
    ("TSP-v0", 200, 600, {"parenting": 2}, 220),              # SPARSE N > 64: the cut-vertex pruning is not vacuous (VERDICT r01)
    ("DensestSubgraph-v0", 500, 4000, {"parenting": 1}, 60),  # the bench's Densest shape
    ("MaxIndependentSet-v0", 200, 600, {}, 210),
    ("DensestSubgraph-v0", 80, 300, {"parenting": 1}, 40),
    ("DensestSubgraph-v0", 80, 300, {"parenting": 0}, 40),
    ("MulticastRouting-v0", 120, 600, {"parenting": 4, "n_dests": 5}, 80),
    ("MulticastRouting-v0", 60, 200, {"parenting": 2, "n_dests": 3}, 60),
    ("MulticastRouting-v0", 40, 120, {"parenting": 1, "n_dests": 3}, 20),
    ("DistributionCenter-v0", 120, 500, {"parenting": 2}, 40),
    ("DistributionCenter-v0", 90, 300, {"parenting": 1, "max_distance": 1.2}, 40),
    ("DistributionCenter-v0", 80, 1500, {"parenting": 2, "target_count": 20}, 30),   # degree ~37 > 32: prefixes continue past the fixed-stride rows (dc_rows)
    ("PerishableProductDelivery-v0", 40, 100, {"n_products": 3, "parenting": 1}, 400),      # SURVEY 8(f4)
    ("PerishableProductDelivery-v0", 300, 900, {"n_products": 5, "parenting": 1}, 300),
    ("PerishableProductDelivery-v0", 12, 20, {"n_products": 5, "parenting": 1, "weighted": False}, 3200),   # runs into max_steps = N * P * 50
]


@pytest.mark.parametrize("cfg", CONFIGS, ids=["%s-N%d-E%d-%s" % (c[0][:-3], c[1], c[2], "".join("%s%s" % (k[0], v) for k, v in c[3].items())) for c in CONFIGS])
@pytest.mark.parametrize("path", ["auto", "warp"])
def test_random_rollout_matches_oracle(cfg, path):
    env_id, N, E, kw, T = cfg
    if path == "warp" and not cu.has_fast_path(env_id, N, kw.get("parenting")):
        pytest.skip("warp-per-env is already the auto path here")
    B, seed = (150 if N < 1000 else 20), 7   # not a multiple of the 128-env block of the lane kernels
    env = BatchedGraphEnv(env_id, B, N, E, auto_reset=True, force_warp=(path == "warp"), **kw)
    p = env.params
    inst = []
    for b in range(B):
        random.seed(1000 + b)
        np.random.seed(1000 + b)
        inst.append(generate_instance(env_id, p))
    u01 = None
    if env_id == "MulticastRouting-v0":
        u01 = torch.tensor([i.u01 for i in inst], dtype=torch.float64, device="cuda")
    env.load_instances(inst)
    if u01 is not None:
        env.finalize_graphs(u01=u01)
        md = env.t["max_dist32"].cpu().numpy()
        for b, i in enumerate(inst):
            i.max_distance = float(md[b])
    oenvs = [cu.oracle_from_instance(env_id, i, p) for i in inst]
    if env_id == "MulticastRouting-v0":  # max_distance itself: fp64 SSSP extremes, multicast_routing.py:98-103
        for b, (i, oe) in enumerate(zip(inst, oenvs)):
            dist = oe.sssp(0)
            ft = max(dist[t] for t in i.dests)
            exp = np.float32(i.u01 * (dist.max() - ft) + ft)
            assert np.float32(md[b]) == exp
    info = env.reset()
    torch.cuda.synchronize()
    masks = [oe.mask(reset_patch=True) for oe in oenvs]
    np.testing.assert_array_equal(info["mask"].cpu().numpy(), np.stack(masks))
    for t in range(T):
        acts = env.sample_actions(seed, t).cpu().numpy()
        for b in range(B):
            assert acts[b] == orc.sample_action(masks[b], seed, b, t), "sampler parity"
        reward, done, info = env.step(env.actions_dev)
        torch.cuda.synchronize()
        reward = reward.cpu().numpy(); done = done.cpu().numpy()
        solved = info["solved"].cpu().numpy(); status = info["status"].cpu().numpy()
        cost = info["solution_cost"].cpu().numpy(); gmask = info["mask"].cpu().numpy()
        for b, oe in enumerate(oenvs):
            o = oe.step(int(acts[b]))
            tag = "%s env %d step %d" % (env_id, b, t)
            assert status[b] == o["status"], tag
            if o["status"] != 0:
                # only reachable with LongestPath parenting=3, whose late-game mask re-enables non-neighbours
                # that step() then rejects (longest_path.py:141-143 vs :153): AssertionError, state unchanged
                assert env_id == "LongestPath-v0" and kw.get("parenting") == 3, tag
                np.testing.assert_array_equal(gmask[b], masks[b], err_msg="mask " + tag)
                continue
            assert bool(done[b]) == o["done"], tag
            assert int(solved[b]) == o["solved"], tag
            assert abs(reward[b] - o["reward"]) <= 1e-5 * max(1.0, abs(o["reward"])), (tag, reward[b], o["reward"])
            if np.isnan(o["solution_cost"]):
                assert np.isnan(cost[b]), tag
            else:
                assert abs(cost[b] - o["solution_cost"]) <= 1e-5 * max(1.0, abs(o["solution_cost"])), tag
            if o["done"]:
                oe.reset_state()
                masks[b] = oe.mask(reset_patch=True)
            elif o["has_mask"]:
                masks[b] = o["mask"]
            np.testing.assert_array_equal(gmask[b], masks[b], err_msg="mask " + tag)
    # observation wire format at the end of the rollout (features off => zeros on both sides)
    obs = env.obs_flat().cpu().numpy()
    for b, oe in enumerate(oenvs):
        np.testing.assert_array_equal(obs[b], oe.obs(), err_msg="obs env %d" % b)
    st = env.stats().cpu().numpy()
    assert st[0] >= 1 or T < 30 or N > 200


@pytest.mark.parametrize("cfg", [("LongestPath-v0", 50, 200, {"parenting": 2}), ("ShortestPath-v0", 10, 20, {}),
                                 ("TSP-v0", 40, 120, {"parenting": 2}), ("SteinerTree-v0", 100, 500, {"n_dests": 99}),
                                 ("MulticastRouting-v0", 120, 600, {"parenting": 4, "n_dests": 5}),
                                 ("DistributionCenter-v0", 120, 500, {"parenting": 2})],
                         ids=lambda c: c[0][:-3])
def test_fused_sampled_step_equals_sample_then_step(cfg):
    """ge_step_sampled (one launch) == ge_sample_actions + ge_step, bit for bit, including the per-env
    clock that lets captured graphs draw fresh actions."""
    env_id, N, E, kw = cfg
    B, T = 300, 50
    envs = []
    for fused in (False, True):
        e = BatchedGraphEnv(env_id, B, N, E, auto_reset=True, **kw)
        e.generate(seed=21)
        e.reset()
        e.enable_env_clock()
        acts = []
        for t in range(T):
            if fused:
                acts.append(e.step_sampled(5, 0).clone())
            else:
                e.sample_actions(5, 0)
                acts.append(e.actions_dev.clone())
                e.step_async(e.actions_dev)
        torch.cuda.synchronize()
        envs.append((e, torch.stack(acts)))
    (a, aa), (b, ab) = envs
    assert torch.equal(aa, ab)
    assert len(torch.unique(aa[:, 0])) > 1, "the per-env clock must vary the draws"
    for name in ("traj", "acc", "mask_bits", "node_bits", "head", "cost"):
        assert torch.equal(a.t[name], b.t[name]), name
    assert torch.equal(a.env_steps, b.env_steps) and int(a.env_steps.min()) == T


def test_host_stepper_graph_replay_matches_direct_calls():
    """ge_step_host on a side stream is captured once and replayed as a CUDA graph: identical results to the
    uncaptured path (default stream) step after step."""
    B, T = 300, 40
    logs = []
    for use_side in (False, True):
        e = BatchedGraphEnv("LongestPath-v0", B, 50, 200, parenting=2, auto_reset=True)
        e.generate(seed=41)
        e.reset()
        blk, h_rew, h_flg, h_cost, h_bits = e.host_io()
        h_act = torch.zeros(B, dtype=torch.int32).pin_memory()
        side = torch.cuda.Stream() if use_side else None
        torch.cuda.synchronize()
        stepper = e.host_stepper(h_act, h_rew, h_flg, h_cost, None, h_bits, stream=side)
        log = []
        for t in range(T):
            h_act.copy_(e.sample_actions(3, t).cpu())
            torch.cuda.synchronize()
            stepper()
            assert torch.equal(h_bits, e.t["mask_bits"].cpu())
            log.append((h_rew.clone(), h_flg.clone(), h_bits.clone()))
        logs.append(log)
    for (r0, f0, m0), (r1, f1, m1) in zip(*logs):
        assert torch.equal(r0, r1) and torch.equal(f0, f1) and torch.equal(m0, m1)


@pytest.mark.parametrize("cfg", [("LongestPath-v0", 50, 200, {"parenting": 2}), ("MulticastRouting-v0", 60, 200, {"parenting": 4, "n_dests": 3}),
                                 ("DistributionCenter-v0", 90, 300, {"parenting": 2}), ("TSP-v0", 70, 300, {"parenting": 1})],
                         ids=lambda c: c[0][:-3])
def test_obs_graph_equals_devectorized_flat_obs(cfg):
    """ge_obs_graph == utils.devectorize_graph(ge_obs_flat) (utils.py:14-23), indices as exact int64."""
    from graphenvs_b200 import utils
    env_id, N, E, kw = cfg
    env = BatchedGraphEnv(env_id, 40, N, E, auto_reset=True, structural_features=True, **kw)
    env.generate(seed=8)
    env.reset()
    for t in range(7):
        env.step_sampled(2, t)
    flat = env.obs_flat(3, 20)
    x, ea, ei = env.obs_graph(3, 20)
    fx, fe, fi = utils.devectorize_graph(flat, env_id, n_nodes=N, n_edges=E)
    assert torch.equal(x, fx) and torch.equal(ea, fe) and torch.equal(ei, fi) and ei.dtype == torch.int64


@pytest.mark.parametrize("cfg", [("LongestPath-v0", 50, 200, {"parenting": 2}), ("TSP-v0", 100, 400, {"parenting": 2}),
                                 ("SteinerTree-v0", 60, 150, {"n_dests": 5}), ("MulticastRouting-v0", 60, 200, {"parenting": 4, "n_dests": 3}),
                                 ("DistributionCenter-v0", 90, 300, {"parenting": 2}), ("MaxIndependentSet-v0", 200, 600, {})],
                         ids=lambda c: c[0][:-3])
def test_pipelined_host_step_equals_single_pass(cfg):
    """ge_step_host_pipelined (slices on parallel graph branches, kernel-driven write-back into the four pinned host
    arrays) returns what ge_step_host returns, step after step, for every kernel family; B is not a multiple of the
    slice size, so the last slice is ragged."""
    env_id, N, E, kw = cfg
    B, T = 1000, 30
    logs = []
    for mode in ("single", "pipelined", "compact", "streamed"):
        pipelined = mode != "single"
        e = BatchedGraphEnv(env_id, B, N, E, auto_reset=True, **kw)
        e.generate(seed=33)
        e.reset()
        if mode == "streamed":   # chunks = 0: one step kernel + the concurrent write-back fed by ge_batch.progress (lane families; two slices elsewhere)
            assert bool(e.lib.ge_progress_supported(__import__("ctypes").byref(e.desc))) == (env_id in ("LongestPath-v0", "DistributionCenter-v0"))
        if mode == "compact":    # ge_step_host_compact: one flag byte per env, float32 solution_cost
            h_rew, h_flg, h_cost, h_bits = e.host_io_compact()
        else:
            blk, h_rew, h_flg, h_cost, h_bits = e.host_io()
        h_act = torch.zeros(B, dtype=torch.int32).pin_memory()
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        xbuf = torch.zeros((B, N, e.F), dtype=torch.float32, device="cuda") if pipelined else None
        stepper = e.host_stepper(h_act, h_rew, h_flg, h_cost, None, h_bits, stream=side, pipelined=pipelined, chunks=0 if mode == "streamed" else 3,
                                 obs_x=xbuf, compact=(mode == "compact"))
        log = []
        for t in range(T):
            h_act.copy_(e.sample_actions(9, t).cpu())
            torch.cuda.synchronize()
            stepper()
            if pipelined:   # ge_batch.obs_x: the call also rewrote the observation's node columns, slice by slice
                assert torch.equal(xbuf, e.obs_nodes()), "obs_x must hold the node columns of the state after the step"
            assert torch.equal(h_bits, e.t["mask_bits"].cpu()), "host mask must equal the device mask after the call"
            assert torch.equal(h_rew, e.reward.cpu())
            if mode == "compact":
                done, solved, status, has_mask = BatchedGraphEnv.unpack_flags8(h_flg)
                flg = torch.from_numpy(np.stack([done.astype(np.uint8), solved.astype(np.int8).view(np.uint8), status, has_mask.astype(np.uint8)], axis=1))
                assert torch.equal(flg, e.flags.cpu()), "flag byte must decode to the four flag fields"
                assert torch.equal(torch.nan_to_num(h_cost, nan=-7.0), torch.nan_to_num(e.solution_cost.float().cpu(), nan=-7.0))
                log.append((h_rew.clone(), flg, e.solution_cost.cpu().clone(), h_bits.clone()))
            else:
                assert torch.equal(h_flg, e.flags.cpu())
                log.append((h_rew.clone(), h_flg.clone(), h_cost.clone(), h_bits.clone()))
        logs.append((log, e.t["traj"].clone(), e.t["acc"].clone()))
        del stepper
    (l0, t0, a0) = logs[0]
    for (l1, t1, a1) in logs[1:]:
        for (r0, f0, c0, m0), (r1, f1, c1, m1) in zip(l0, l1):
            assert torch.equal(r0, r1) and torch.equal(f0, f1) and torch.equal(m0, m1)
            assert torch.equal(torch.nan_to_num(c0, nan=-7.0), torch.nan_to_num(c1, nan=-7.0))
        assert torch.equal(t0, t1) and torch.equal(a0, a1)


def test_sliced_descriptors_step_like_the_full_batch():
    """ge_batch_slice: stepping the three slices of a batch one after the other == stepping the batch (same memory)."""
    import ctypes as C
    from graphenvs_b200 import _native
    for env_id, N, E, kw in [("LongestPath-v0", 50, 200, {"parenting": 2}), ("MulticastRouting-v0", 60, 200, {"parenting": 4, "n_dests": 3})]:
        B, T = 700, 25
        full = BatchedGraphEnv(env_id, B, N, E, auto_reset=True, **kw)
        part = BatchedGraphEnv(env_id, B, N, E, auto_reset=True, **kw)
        for e in (full, part):
            e.generate(seed=5)
            e.reset()
        cuts = [(0, 256), (256, 320), (576, 124)]
        descs = [part.slice_desc(lo, n) for lo, n in cuts]
        for t in range(T):
            acts = full.sample_actions(4, t).clone()
            full.step_async(acts)
            for (lo, n), dsc in zip(cuts, descs):
                out = _native.StepOut(part.reward[lo:].data_ptr(), part.flags[lo:].data_ptr(), part.solution_cost[lo:].data_ptr())
                _native.check(part.lib.ge_step(C.byref(dsc), acts[lo:].data_ptr(), C.byref(out), part._stream()))
            torch.cuda.synchronize()
            assert torch.equal(full.reward, part.reward) and torch.equal(full.flags, part.flags)
        for name in ("traj", "acc", "mask_bits", "node_bits", "cost"):
            assert torch.equal(full.t[name], part.t[name]), name


def test_obs_nodes_is_the_x_tensor_of_obs_graph():
    for env_id, N, E, kw in [("LongestPath-v0", 50, 200, {"parenting": 2}), ("DistributionCenter-v0", 90, 300, {"parenting": 2}),
                             ("MulticastRouting-v0", 60, 200, {"parenting": 4, "n_dests": 3}), ("TSP-v0", 33, 100, {"parenting": 1})]:
        env = BatchedGraphEnv(env_id, 50, N, E, auto_reset=True, structural_features=True, **kw)
        env.generate(seed=8)
        env.reset()
        for t in range(5):
            env.step_sampled(2, t)
        x, ea, ei = env.obs_graph()
        assert torch.equal(env.obs_nodes(), x)
        assert torch.equal(env.obs_nodes(7, 11), x[7:18])
        name = env.step_kernel_name(sampled=True)
        assert name.endswith(">") and "step_kernel<" in name


@pytest.mark.parametrize("shape", [(120, 500), (80, 1500), (500, 4000)], ids=["sparse", "degree>32", "cfg5"])
def test_distribution_center_fixed_stride_rows_equal_general_family(shape):
    """The dedicated DistributionCenter kernel, whose cutoff search reads ge_batch.dc_rows (weight-sorted rows at a fixed
    128-byte stride, prefixes longer than 32 entries continued in dc_edges), gives the same trajectories, masks and covered
    sets as the general warp-per-env family (GE_FLAG_FORCE_WARP), whose search walks the CSR rows."""
    N, E = shape
    B, T = 256, 40
    envs = []
    for force_warp in (False, True):
        e = BatchedGraphEnv("DistributionCenter-v0", B, N, E, parenting=2, target_count=min(100, N // 4), max_distance=1, auto_reset=True,
                            force_warp=force_warp)
        e.generate(seed=21)
        e.reset()
        assert e.step_kernel_name().startswith("step_kernel<" if force_warp else "dc_step_kernel")
        for t in range(T):
            e.step_sampled(4, t)
        torch.cuda.synchronize()
        envs.append(e)
    a, b = envs
    assert "dc_rows" in a.t
    assert torch.equal(a.t["row_ptr"], b.t["row_ptr"]) and torch.equal(a.t["col"], b.t["col"]), "both batches must hold the same graphs"
    if N == 80:
        deg = (a.t["row_ptr"][:, 1:N + 1] - a.t["row_ptr"][:, :N]).max().item()
        assert deg > 32, "this shape is meant to overflow the 32-entry rows"
    for k in ("traj", "mask_bits", "node_bits", "node_bits2", "cost", "acc", "done"):
        assert torch.equal(a.t[k], b.t[k]), k
