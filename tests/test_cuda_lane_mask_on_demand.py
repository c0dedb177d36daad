"""GPU: the lane-per-env family (csrc/ge_lane.cu, N <= 64) keeps only the packed mask current.  Its reset and step
kernels never write the byte view `mask_bytes`; `env.mask`, the `h_mask` of the host step and a state load expand it on
demand because ge_mask_bytes_current() is 0.  When an episode ends, the step loads its statistics rows (acc) together
before it stores them, with the same arithmetic as the general family."""
import ctypes as C

import numpy as np
import pytest
import torch

from graphenvs_b200 import BatchedGraphEnv, _native

pytestmark = pytest.mark.gpu

KINDS = [
    ("ShortestPath-v0", {}),
    ("LongestPath-v0", {"parenting": 0}),
    ("LongestPath-v0", {"parenting": 1}),
    ("LongestPath-v0", {"parenting": 2}),
    ("LongestPath-v0", {"parenting": 3}),
    ("TSP-v0", {"parenting": 1}),
    ("TSP-v0", {"parenting": 2}),
    ("MaxIndependentSet-v0", {}),
    ("DensestSubgraph-v0", {"parenting": 1}),
]
CASES = [(env_id, N, 3 * N, kw) for env_id, kw in KINDS for N in (10, 33, 50, 64)]
IDS = ["%s-N%d%s" % (c[0][:-3], c[1], "".join("-%s%s" % (k[0], v) for k, v in c[3].items())) for c in CASES]
FILL = 0xAB
B = 256


def steps_for(N):
    """Steps that cross an auto-reset in every kind: a MaxIndependentSet episode takes up to N steps."""
    return N + 10


def unpacked(bits, A):
    """bool[B, A] of a packed int32[B, AW] mask (bit j of word w = action 32 w + j)."""
    shifts = torch.arange(32, device=bits.device, dtype=torch.int32)
    return ((bits.unsqueeze(-1) >> shifts) & 1).reshape(bits.shape[0], -1)[:, :A].bool()


def lane_batch(env_id, N, E, kw, seed=5):
    env = BatchedGraphEnv(env_id, B, N, E, auto_reset=True, **kw)
    env.generate(seed=seed)
    env.enable_env_clock()
    assert env.step_kernel_name(sampled=True).startswith("lane_step_kernel<"), env.step_kernel_name(sampled=True)
    assert "mask_bytes" in env.t
    return env


def native_reset(env):
    """ge_reset without BatchedGraphEnv.reset()'s info dict, which reads env.mask and so expands the byte view."""
    _native.check(env.lib.ge_reset(C.byref(env.desc), None, env._stream()))


def assert_mask(env, what):
    """env.mask equals the packed mask unpacked, bit for bit, although the byte view held FILL before."""
    m = env.mask
    assert m.dtype == torch.bool
    assert torch.equal(m, unpacked(env.t["mask_bits"], env.desc.A)), what
    env.t["mask_bytes"].fill_(FILL)       # a later check that skipped the expansion would see FILL, not a stale copy


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_lane_steps_leave_the_byte_view_alone(case):
    env_id, N, E, kw = case
    env = lane_batch(env_id, N, E, kw)
    env.t["mask_bytes"].fill_(FILL)
    native_reset(env)                     # lane_reset_kernel
    for t in range(steps_for(N)):
        env.step_sampled(3, t)            # lane_step_kernel<*, 1>, auto-reset included
    torch.cuda.synchronize()
    assert int(env.t["acc"][0].sum().item()) > 0, "the rollout must cross at least one auto-reset"
    assert bool((env.t["mask_bytes"] == FILL).all()), "a lane kernel wrote the byte view"
    assert env.lib.ge_mask_bytes_current(C.byref(env.desc)) == 0


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_lane_mask_is_expanded_on_demand(case):
    env_id, N, E, kw = case
    env = lane_batch(env_id, N, E, kw)
    env.t["mask_bytes"].fill_(FILL)
    native_reset(env)
    assert_mask(env, "after reset")
    T = steps_for(N)
    for t in range(T):
        env.step_sampled(4, t)
        assert_mask(env, "after step %d" % t)
    assert int(env.t["acc"][0].sum().item()) > 0

    # load_states: the state load does not rebuild the byte view for this family, env.mask does
    saved_bits = env.t["mask_bits"].clone()
    saved = env.save_states()
    for t in range(T, T + 6):
        env.step_sampled(4, t)
    env.t["mask_bytes"].fill_(FILL)
    env.load_states(saved)
    torch.cuda.synchronize()
    assert bool((env.t["mask_bytes"] == FILL).all()), "the state load rebuilt the byte view"
    assert torch.equal(env.t["mask_bits"], saved_bits)
    assert_mask(env, "after load_states")

    # the host step's byte mask (h_mask): direct on the default stream, then captured and replayed on a side stream
    A, AP, AW = env.desc.A, env.desc.AP, env.desc.AW
    h_act = torch.zeros(B, dtype=torch.int32).pin_memory()
    h_rew = torch.zeros(B, dtype=torch.float32).pin_memory()
    h_flg = torch.zeros((B, 4), dtype=torch.uint8).pin_memory()
    h_cost = torch.zeros(B, dtype=torch.float64).pin_memory()
    h_mask = torch.zeros((B, AP), dtype=torch.uint8).pin_memory()
    h_bits = torch.zeros((B, AW), dtype=torch.int32).pin_memory()
    side = torch.cuda.Stream()
    for t, stream in ((40, None), (41, side), (42, side), (43, side)):
        env.sample_actions(6, t)
        h_act.copy_(env.actions_dev)
        env.t["mask_bytes"].fill_(FILL)
        torch.cuda.synchronize()
        if stream is None:
            env.step_host(h_act, h_rew, h_flg, h_cost, h_mask, h_bits)
        else:
            with torch.cuda.stream(stream):
                env.step_host(h_act, h_rew, h_flg, h_cost, h_mask, h_bits)
        torch.cuda.synchronize()
        # (LongestPath parenting 3 offers actions that its step then rejects, so the status is not checked here)
        want = unpacked(env.t["mask_bits"], A).cpu()
        assert torch.equal(unpacked(h_bits, A), want), "h_mask_bits, host step at t=%d" % t
        assert torch.equal(h_mask[:, :A].bool(), want), "h_mask, host step at t=%d" % t
        assert not bool(h_mask[:, A:].any()), "h_mask padding"


STATS_CASES = [
    ("LongestPath-v0", 50, 200, {"parenting": 2, "weighted": True}, 4096, 300),     # cfg2 shape: lane_step_kernel<1, *>
    ("ShortestPath-v0", 10, 20, {"weighted": True}, 4096, 200),                    # cfg1 shape: lane_step_kernel<0, *>
]


@pytest.mark.parametrize("case", STATS_CASES, ids=["cfg2-LongestPath-N50-p2", "cfg1-ShortestPath-N10"])
def test_lane_statistics_equal_general_family(case):
    """Every row of acc, and stats(), after many episodes: the lane kernel against a force_warp twin stepped with the same
    actions, bit for bit."""
    env_id, N, E, kw, n, T = case
    envs = []
    for force_warp in (False, True):
        e = BatchedGraphEnv(env_id, n, N, E, auto_reset=True, force_warp=force_warp, **kw)
        e.generate(seed=23)
        e.reset()
        envs.append(e)
    lane, warp = envs
    lane.enable_env_clock()
    assert lane.step_kernel_name(sampled=True).startswith("lane_step_kernel<")
    assert warp.step_kernel_name().startswith("step_kernel<")
    assert torch.equal(lane.t["row_ptr"], warp.t["row_ptr"]) and torch.equal(lane.t["col"], warp.t["col"]), "both batches must hold the same graphs"
    for t in range(T):
        lane.step_sampled(8, t)
        warp.step_async(lane.actions_dev)
    torch.cuda.synchronize()
    episodes = lane.t["acc"][0].sum().item()
    assert episodes > 4 * n, "the rollout must end many episodes (%d)" % episodes
    for k in range(4):
        assert torch.equal(lane.t["acc"][k].view(torch.int64), warp.t["acc"][k].view(torch.int64)), "acc[%d]" % k
    for k in ("traj", "mask_bits", "done", "head"):
        assert torch.equal(lane.t[k], warp.t[k]), k
    # stats() adds per-block partial sums with atomics in whatever order the blocks finish: the episode and solved counts are
    # exact, the reward and cost sums agree up to that order
    s_lane, s_warp = lane.stats().cpu().numpy().copy(), warp.stats().cpu().numpy().copy()
    assert np.array_equal(s_lane[:2], s_warp[:2]), "stats() counts"
    assert s_lane[0] == episodes
    assert np.allclose(s_lane[2:], s_warp[2:], rtol=1e-12, atol=0), "stats() sums"
    assert np.allclose(s_lane, lane.t["acc"].sum(dim=1).cpu().numpy(), rtol=1e-12, atol=0)
