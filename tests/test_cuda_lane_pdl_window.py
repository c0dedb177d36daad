"""GPU: the lane-per-env step (csrc/ge_lane.cu) reaches the dynamic state before griddepcontrol.wait through L2 only -- L2
prefetches of this env's state, and in the sampled kernel a draw guessed from L2 loads whose edge weight it prefetches -- and
settles the statistics rows (acc) with fp64 reductions.  None of that may change a result.  Under programmatic dependent
launch every lane kind ends bit-identical to a plain-launch twin in state, outputs, trajectory checksums and all four acc rows:
- one batch stepped back to back on one stream, where the previous launch is still writing the state a guess is made from;
- the same with a state load between steps that takes every env one step back, rewriting the state under the next step's wait;
- the benchmark's schedule, R batches rotating over C stream chains, where the guess is right."""
import pytest
import torch

from graphenvs_b200 import BatchedGraphEnv
from graphenvs_b200.batch import STATE_DYNAMIC, SliceStreams

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
B = 256
SEED = 13
STATE = ("node_bits", "node_bits2", "head", "cost", "counters", "done", "mask_bits", "traj", "acc")


def steps_for(N):
    """Enough steps for every env to finish at least one episode: a MaxIndependentSet or TSP episode takes up to N + 1."""
    return 2 * N + 10


def make(case, env_id0=0):
    env_id, N, E, kw = case
    env = BatchedGraphEnv(env_id, B, N, E, auto_reset=True, env_id0=env_id0, **kw)
    env.generate(seed=21 + env_id0)
    env.reset()
    env.enable_env_clock()
    assert env.step_kernel_name(sampled=True).startswith("lane_step_kernel<"), env.step_kernel_name(sampled=True)
    return env


def bits(t):
    """Bit pattern of a tensor (NaN solution costs compare equal to themselves)."""
    return t.contiguous().view(torch.uint8)


def assert_twins(ref, env, what):
    torch.cuda.synchronize()
    for k in STATE:
        if k in ref.t:
            assert torch.equal(bits(ref.t[k]), bits(env.t[k])), "%s: %s differs from the plain-launch twin" % (what, k)
    assert torch.equal(ref.env_steps, env.env_steps), "%s: env_steps" % what
    for name in ("reward", "flags", "solution_cost", "actions_dev"):
        assert torch.equal(bits(getattr(ref, name)), bits(getattr(env, name))), "%s: %s" % (what, name)


def assert_every_env_reset(env):
    finished = env.t["acc"][0] >= 1
    if env.env_id == "LongestPath-v0" and env.desc.parenting == 3:
        # Once few nodes are left, parenting 3 offers every remaining node but the step rejects a non-neighbour of the head as
        # invalid (state unchanged): an env whose mask holds only non-neighbours never moves again.  Most envs still finish.
        assert float(finished.float().mean()) >= 0.5, "too few envs finished an episode: the auto-reset path went untested"
    else:
        assert bool(finished.all()), "some env finished no episode: the auto-reset path went untested"


def run_on_side_stream(fn, graph):
    """fn() eagerly on a side stream, or captured there into one CUDA graph and replayed once (PDL edges between nodes)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    if graph:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            fn()
        g.replay()
    else:
        with torch.cuda.stream(side):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()


@pytest.mark.parametrize("sampled", [True, False], ids=["sampled", "actions"])
@pytest.mark.parametrize("graph", [False, True], ids=["eager", "graph"])
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_one_batch_back_to_back(case, graph, sampled):
    T = steps_for(case[1])

    def steps(env):
        for t in range(T):
            if sampled:
                env.step_sampled(SEED, t)
            else:
                env.sample_actions(SEED, t)
                env.step_async(env.actions_dev)

    ref = make(case)
    steps(ref)
    env = make(case)
    env.enable_pdl()
    run_on_side_stream(lambda: steps(env), graph)
    assert_twins(ref, env, "back to back")
    assert_every_env_reset(ref)


@pytest.mark.parametrize("graph", [False, True], ids=["eager", "graph"])
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_state_loads_between_steps(case, graph):
    T = steps_for(case[1]) * 3 // 2     # one step in three is taken back

    def steps(env, buf):
        for t in range(T):
            if t % 3 == 1:
                env.save_states(out=buf)
            env.step_sampled(SEED, t)
            if t % 3 == 1:      # every env back to its own state before this step, right before the next step's wait window;
                env.load_states(buf, what=STATE_DYNAMIC)   # the clock runs on, so the next draw differs

    ref = make(case)
    steps(ref, ref.save_states())
    env = make(case)
    env.enable_pdl()
    buf = env.save_states()
    run_on_side_stream(lambda: steps(env, buf), graph)
    assert_twins(ref, env, "state loads between steps")
    assert_every_env_reset(ref)


@pytest.mark.parametrize("graph", [False, True], ids=["eager", "graph"])
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_batches_rotating_over_stream_chains(case, graph):
    R, C_ = 3, 4
    T = steps_for(case[1])
    refs = [make(case, env_id0=r * B) for r in range(R)]
    for ref in refs:
        for t in range(T):
            ref.step_sampled(SEED, t)
    envs = [make(case, env_id0=r * B) for r in range(R)]
    for e in envs:
        e.enable_pdl()
    streams = [torch.cuda.Stream() for _ in range(C_)]
    sl = [SliceStreams(e, C_, streams=streams) for e in envs]

    def steps():
        sl[0].fork()
        for i in range(R * T):
            sl[i % R].step_sampled(SEED, i // R)
        sl[0].join()

    run_on_side_stream(steps, graph)
    for r in range(R):
        assert_twins(refs[r], envs[r], "batch %d of %d rotating over %d chains" % (r, R, C_))
        assert_every_env_reset(refs[r])
