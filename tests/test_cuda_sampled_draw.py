"""GPU: the action draw inside the fused step (ge_step_sampled) against an exact reference of that draw, per sampler variant,
and at every benched workload stepped the way bench.py steps it.

Every step-kernel family carries its own copy of the draw.  All of them must pick the r-th set bit of the env's packed mask,
r = mix32(seed, env_id0 + b, t + env_steps[b]) * popcount >> 32, as ge_sample_actions and the oracle's oenv_sample_action do:

  lane family (ge_lane.cu)          lane_sample: one lane per env, the mask as one 64-bit register (N <= 64)
  group family (ge_group.cu)        group_step_kernel: G = 8 / 16 / 32 lanes, one mask word per lane (64 < N <= 1024)
  incremental tree (ge_incr.cu)     incr_tree_step_kernel, total from counters[1], one of three walks:
                                      group_sample_regs (ge_common.cuh): the whole mask in registers, AW <= 4 G
                                      group_sample_chunks: the 16 chunk popcounts of mask_cnt, then one chunk (mask_cnt, G >= 16)
                                      group_sample (ge_common.cuh): G words at a time
  incremental MIS (ge_incr.cu)      incr_mis_step_kernel: a word walk, total = N - counters[0]
  DistributionCenter (ge_dc.cu)     dc_step_kernel: one mask word per lane of a warp
  Perishable (ge_ppd.cu)            ppd_lane_step_kernel (64-bit lane draw, N <= 64), ppd_step_kernel (warp_sample)
  general family (ge_api.cu)        step_kernel: warp_sample (ge_common.cuh)

The incremental draws trust state the kernels keep up to date -- counters[1], N - counters[0] and the 16-bit chunk counts of
mask_cnt -- so those are checked against the mask they describe after every checked step.  The reference computes the
popcount from the mask itself, never from that state."""
import functools
import gc
import os
import random
import sys
import traceback

import numpy as np
import pytest
import torch

import cuda_util as cu
from graphenvs_b200 import BatchedGraphEnv
from graphenvs_b200.batch import SliceStreams
from graphenvs_b200.instances import generate_instance
from oracle import oracle as orc

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402

pytestmark = pytest.mark.gpu

U32 = 0xFFFFFFFF
STATE = ("mask_bits", "mask_cnt", "counters", "head", "node_bits", "node_bits2", "edge_bits", "dist32", "bestkey", "cost", "done",
         "traj", "acc")
_POP8 = [bin(i).count("1") for i in range(256)]


# ------------------------------------------------------------------ exact reference of the draw
def np_mix32(seed, env, t):
    """ge_common.cuh:mix32 in numpy uint64 arithmetic (wrapping); arguments broadcast."""
    with np.errstate(over="ignore"):
        seed, env, t = np.uint64(seed), np.asarray(env, dtype=np.uint64), np.asarray(t, dtype=np.uint64)
        z = seed + np.uint64(0x9E3779B97F4A7C15) * (env * np.uint64(0x100000001) + ((t << np.uint64(32)) | np.uint64(0x5bd1e995)))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
        return z >> np.uint64(32)


def _row_blocks(B, AW, words=1 << 22):
    """Env ranges of at most `words` mask words: bounds the scratch of the reference and the invariant checks
    (cfg5 Multicast is 131,072 x 250 words)."""
    per = max(1, words // max(AW, 1))
    return [(lo, min(B, lo + per)) for lo in range(0, B, per)]


def word_popcounts(words):
    """int64 [n, AW] popcount of every word of int32 [n, AW], through a byte lookup table."""
    n, AW = words.shape
    lut = torch.tensor(_POP8, dtype=torch.int64, device=words.device)
    return lut[words.contiguous().view(torch.uint8).long()].view(n, AW, 4).sum(2)


def expected_draw(mask_bits, env_steps, env_id0, seed, t):
    """Action the in-kernel draw must pick for every env: the r-th set bit of mask_bits[b], r = mix32(seed, env_id0 + b,
    t + env_steps[b]) * total >> 32 with total the popcount of the row; -1 for an empty row.  int64 [B] on the mask's device."""
    B, AW = mask_bits.shape
    dev = mask_bits.device
    steps = np.zeros(B, np.uint64) if env_steps is None else env_steps.cpu().numpy().astype(np.int64).astype(np.uint64) & np.uint64(U32)
    env = (np.arange(B, dtype=np.uint64) + np.uint64(env_id0)) & np.uint64(U32)
    mix = np_mix32(seed, env, (np.uint64(t & U32) + steps) & np.uint64(U32))
    out = torch.empty(B, dtype=torch.int64, device=dev)
    bit = torch.arange(32, device=dev)
    for lo, hi in _row_blocks(B, AW):
        words = mask_bits[lo:hi]
        pc = word_popcounts(words)
        cum = pc.cumsum(1)
        total = cum[:, -1]
        r = (mix[lo:hi] * total.cpu().numpy().astype(np.uint64)) >> np.uint64(32)    # < 2^64: mix < 2^32, total < 2^32
        r = torch.from_numpy(r.astype(np.int64)).to(dev)
        w = torch.searchsorted(cum, r[:, None], right=True).squeeze(1).clamp_(max=AW - 1)   # first word whose prefix exceeds r
        rank = r - (cum.gather(1, w[:, None]) - pc.gather(1, w[:, None])).squeeze(1)        # r's rank inside that word
        word = words.gather(1, w[:, None]).squeeze(1).long() & U32
        bits = (word[:, None] >> bit) & 1
        pos = ((bits.cumsum(1) == rank[:, None] + 1) & (bits == 1)).int().argmax(1)
        out[lo:hi] = torch.where(total > 0, w * 32 + pos, torch.full_like(w, -1))
    return out


def assert_draws(tag, got, exp, mask, steps):
    bad = torch.nonzero(got.long() != exp).flatten()
    if bad.numel():
        b = int(bad[0])
        pc = int(word_popcounts(mask[b:b + 1]).sum())
        raise AssertionError("%s: %d of %d draws differ from the reference; first env %d: drawn %d, expected %d (env_steps %s, "
                             "popcount %d)" % (tag, bad.numel(), got.numel(), b, int(got[b]), int(exp[b]),
                                               "off" if steps is None else int(steps[b]), pc))


# ------------------------------------------------------------------ what the draws rely on
def check_invariants(env, tag):
    """Full batch: no mask bit at or above A; counters[:, 1] == popcount (incremental tree kernels); popcount ==
    N - counters[:, 0] (incremental MaxIndependentSet); every 16-bit half of mask_cnt == popcount of its chunk of
    ceil(AW / 16) words, the empty trailing chunks included."""
    d = env.desc
    A, AW, B = d.A, d.AW, env.B
    mb = env.t["mask_bits"]
    if A % 32:
        above = (mb[:, AW - 1].long() & U32) >> (A % 32)
        assert not above.any(), "%s: mask bit at or above A = %d in env %d" % (tag, A, int(torch.nonzero(above)[0]))
    name = env.step_kernel_name(sampled=True)
    cnt = env.t.get("mask_cnt")
    CW = (AW + 15) // 16
    for lo, hi in _row_blocks(B, AW):
        pc = word_popcounts(mb[lo:hi])
        total = pc.sum(1)
        c = env.t["counters"][lo:hi].long()
        if name.startswith("incr_tree_step_kernel"):
            bad = torch.nonzero(c[:, 1] != total).flatten()
            assert not bad.numel(), "%s: counters[1] = %d, popcount = %d in env %d" % (
                tag, int(c[bad[0], 1]), int(total[bad[0]]), lo + int(bad[0]))
        if name.startswith("incr_mis_step_kernel"):
            bad = torch.nonzero(total != env.N - c[:, 0]).flatten()
            assert not bad.numel(), "%s: popcount %d != N - counters[0] = %d in env %d" % (
                tag, int(total[bad[0]]), env.N - int(c[bad[0], 0]), lo + int(bad[0]))
        if cnt is not None:
            chunks = torch.nn.functional.pad(pc, (0, 16 * CW - AW)).view(-1, 16, CW).sum(2)
            mc = cnt[lo:hi].long() & U32
            got = torch.stack([mc & 0xFFFF, mc >> 16], 2).view(-1, 16)
            bad = torch.nonzero(got != chunks)
            assert not bad.numel(), "%s: mask_cnt chunk %d of env %d holds %d, its %d words hold %d set bits" % (
                tag, int(bad[0, 1]), lo + int(bad[0, 0]), int(got[bad[0, 0], bad[0, 1]]), CW, int(chunks[bad[0, 0], bad[0, 1]]))


def fused_step_checked(env, seed, t, tag):
    """One eager full-batch ge_step_sampled; the drawn actions against the reference of the mask and clock before it."""
    mask, steps = env.t["mask_bits"].clone(), env.env_steps.clone()
    env.step_sampled(seed, t)
    assert_draws(tag, env.actions_dev, expected_draw(mask, steps, env.desc.env_id0, seed, t), mask, steps)
    assert int(env.flags[:, 2].max()) == 0, "%s: a drawn action was rejected" % tag
    assert torch.equal(env.env_steps, steps + 1), "%s: the env clock did not advance by one" % tag
    check_invariants(env, tag)


def assert_same_state(a, b, tag):
    for k in STATE:
        if k in a.t:
            assert torch.equal(a.t[k], b.t[k]), "%s: %s differs between the fused and the reference-draw batch" % (tag, k)
    assert torch.equal(a.actions_dev, b.actions_dev), "%s: last actions differ" % tag
    assert torch.equal(a.reward, b.reward) and torch.equal(a.flags, b.flags), "%s: last rewards / flags differ" % tag
    assert torch.equal(torch.nan_to_num(a.solution_cost, nan=-7.0), torch.nan_to_num(b.solution_cost, nan=-7.0)), tag


def oracle_slice_matches(env, env_id, inst, lo, T, seed, t0, tag):
    """The oracle steps host copies of envs [lo, lo + len(inst)) T times from the same (seed, global env id, t0 + k)
    draws: trajectory checksums and episode counts bit for bit, reward sums to 1e-5, final masks bit for bit."""
    n = len(inst)
    oenvs = [cu.oracle_from_instance(env_id, i, env.params) for i in inst]
    orc.set_threads(0)
    sr, ep, cs = orc.rollout(oenvs, T, seed, env_id0=env.desc.env_id0 + lo, t0=t0)
    traj = env.t["traj"][lo:lo + n].cpu().numpy().view(np.uint64)
    acc = env.t["acc"][:, lo:lo + n].cpu().numpy()
    np.testing.assert_array_equal(traj, cs, err_msg="%s: trajectory checksums, envs %d.." % (tag, lo))
    np.testing.assert_array_equal(acc[0].astype(np.int64), ep, err_msg="%s: episode counts" % tag)
    np.testing.assert_allclose(acc[2], sr, rtol=1e-5, atol=1e-4, err_msg="%s: reward sums" % tag)
    bits = env.t["mask_bits"][lo:lo + n].cpu().numpy()
    got = np.unpackbits(bits.view(np.uint8), axis=1, bitorder="little")[:, :env.desc.A].astype(bool)
    np.testing.assert_array_equal(got, np.stack([oe.mask(reset_patch=False) for oe in oenvs]), err_msg="%s: final masks" % tag)


def _released(fn):
    """Run fn; on failure drop the locals of its frames, so a failed workload does not keep its batches on the device."""
    @functools.wraps(fn)
    def run(*args, **kw):
        try:
            fn(*args, **kw)
        except BaseException as exc:
            traceback.clear_frames(exc.__traceback__)
            raise
        finally:
            gc.collect()
            torch.cuda.empty_cache()
    return run


# ------------------------------------------------------------------ every benched workload, benched the way bench.py does it
K1 = {"cfg3_mst": 112, "cfg4_tsp_p1": 212, "cfg4_tsp_p2": 212, "cfg4_mis": 212}    # > one episode: N - 1 = 99 / N = 200 steps
K1_DEFAULT = 48
WARMUP = 3          # eager full-batch steps before the capture, as the bench's warm-up
GRAPH_STEPS = 16    # steps per captured graph; K1 - WARMUP is not a multiple, so a remainder graph runs too
J = 8               # eager fused steps checked draw by draw
# envs per oracle slice: sized by the oracle's cost (TSP parenting=2 at N=200: ~850 env-steps/s on 16 host threads)
SLICE_ENVS = {"cfg4_tsp_p2": 2, "cfg5_multicast": 128, "cfg5_distcenter": 128}


def _bench_batch(wl, clock=True, export=()):
    """A batch as measure_workload / measure_streaming build it, rotation batch 1 (env_id0 = B); `export`: (lo, n) ranges
    whose instances are copied out before release_w64(), so the oracle gets the float64 weights."""
    env_id, N, E, kw, B = bench.WORKLOADS[wl][:5]
    env = BatchedGraphEnv(env_id, B, N, E, auto_reset=True, env_id0=B, **kw)
    env.generate(seed=bench.SEED)
    inst = [env.export_instances(lo, n) for lo, n in export]
    env.release_w64()
    env.reset()
    if clock:
        env.enable_env_clock()
    return env, inst


def _require_memory(wl):
    """Skip, naming the workload and the shortfall, when two batches of it do not fit in the free device memory."""
    env_id, N, E, kw, B = bench.WORKLOADS[wl][:5]
    probe = BatchedGraphEnv(env_id, 256, N, E, auto_reset=True, **kw)
    probe.generate(seed=bench.SEED, check=False)
    need = 2.2 * probe.memory_bytes() / 256 * B
    del probe
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if need > free:
        pytest.skip("%s: two batches of %d envs need about %.1f GB, %.1f GB are free (%.1f GB short)"
                    % (wl, B, need / 1e9, free / 1e9, (need - free) / 1e9))


@pytest.mark.parametrize("wl", list(bench.WORKLOADS))
@_released
def test_benched_workload_fused_draw_matches_reference(wl):
    """The benched batch (B, seed, env_id0 of rotation batch 1), stepped as measure_streaming steps it -- PDL, eager
    warm-up, then captured graphs of SliceStreams fork / step / join -- ends in exactly the state of a twin that draws with
    ge_sample_actions and steps with plain launches; J more fused steps are checked draw by draw against the reference,
    with the invariants after each; oracle slices from the start, middle and end replay all K1 + J steps."""
    _require_memory(wl)
    env_id, N, E, kw, B = bench.WORKLOADS[wl][:5]
    seed, k1 = bench.SEED, K1.get(wl, K1_DEFAULT)
    n = SLICE_ENVS.get(wl, 256)
    slices = [(0, n), (B // 2 - n // 2, n), (B - n, n)]
    fz, inst = _bench_batch(wl, export=slices)
    tw, _ = _bench_batch(wl, clock=False)
    name = fz.step_kernel_name(sampled=True)
    assert "SAMPLED=1" in name

    # fused, benched schedule
    fz.enable_pdl()
    chunks = bench.STREAM_CHUNKS.get(wl, 1)
    sl = SliceStreams(fz, chunks) if chunks > 1 else None
    for _ in range(WARMUP):
        fz.step_sampled(seed, 0)
    torch.cuda.synchronize()
    check_invariants(fz, "%s after the warm-up" % wl)

    def capture(steps):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            if sl:
                sl.fork()
            for _ in range(steps):
                (sl or fz).step_sampled(seed, 0)
            if sl:
                sl.join()
        return g
    q, r = divmod(k1 - WARMUP, GRAPH_STEPS)
    assert r, "the schedule is meant to end in a remainder graph"
    graph, tail = capture(GRAPH_STEPS), capture(r)
    for _ in range(q):
        graph.replay()
    tail.replay()
    torch.cuda.synchronize()
    del graph, tail, sl
    fz.enable_pdl(False)

    # twin: ge_sample_actions at t = k (no env clock), then ge_step, plain launches
    for k in range(k1):
        tw.sample_actions(seed, k)
        tw.step_async(tw.actions_dev)
    torch.cuda.synchronize()
    assert bool((fz.env_steps == k1).all()), "%s: every step must be accepted, so the clock is k at step k" % wl
    assert_same_state(fz, tw, "%s (%s), %d steps" % (wl, name, k1))
    check_invariants(fz, "%s after %d steps" % (wl, k1))
    check_invariants(tw, "%s twin after %d steps" % (wl, k1))
    del tw
    torch.cuda.empty_cache()

    for j in range(J):
        fused_step_checked(fz, seed, 0, "%s (%s) step %d" % (wl, name, k1 + j))
    torch.cuda.synchronize()
    for (lo, cnt), ins in zip(slices, inst):
        oracle_slice_matches(fz, env_id, ins, lo, k1 + J, seed, 0, "%s oracle slice" % wl)


# ------------------------------------------------------------------ sampler variants at the dispatch boundaries
def _case(tag, env_id, N, E, kw, B, kernel, T=40, chunks=None, force_warp=False):
    return pytest.param((env_id, N, E, kw, B, kernel, T, chunks, force_warp), id=tag)


LANE_S, LANE_U = "lane_step_kernel<STAGED=1,SAMPLED=1>", "lane_step_kernel<STAGED=0,SAMPLED=1>"
TREE = "incr_tree_step_kernel<SAMPLED=1,G=%d>"
MIS = "incr_mis_step_kernel<SAMPLED=1>"
DC = "dc_step_kernel<SAMPLED=1>"
# chunks: None = no mask_cnt; "regs" = mask_cnt kept but group_sample_regs draws; "chunks" = group_sample_chunks draws
SWEEP = [
    _case("lane-LongestPath-N32-staged", "LongestPath-v0", 32, 80, {"parenting": 2}, 2900, LANE_S),
    _case("lane-TSP-N33-staged", "TSP-v0", 33, 200, {"parenting": 2}, 2900, LANE_S),
    _case("lane-TSP-N64-staged", "TSP-v0", 64, 600, {"parenting": 2}, 2900, LANE_S, T=70),       # bit 63
    _case("lane-ShortestPath-N33", "ShortestPath-v0", 33, 80, {}, 2900, LANE_U),
    _case("lane-LongestPath-N64-p1", "LongestPath-v0", 64, 200, {"parenting": 1}, 2900, LANE_U),
    _case("lane-MIS-N64", "MaxIndependentSet-v0", 64, 200, {}, 2900, LANE_U, T=70),
    _case("lane-Densest-N64", "DensestSubgraph-v0", 64, 300, {"parenting": 1}, 2900, LANE_U),
    _case("group8-ShortestPath-N65", "ShortestPath-v0", 65, 200, {}, 1500, "group_step_kernel<SAMPLED=1,G=8>"),
    _case("group8-TSP-N256", "TSP-v0", 256, 1200, {"parenting": 1}, 1000, "group_step_kernel<SAMPLED=1,G=8>"),
    _case("group16-Densest-N257", "DensestSubgraph-v0", 257, 900, {"parenting": 1}, 1000, "group_step_kernel<SAMPLED=1,G=16>"),
    _case("group16-ShortestPath-N512", "ShortestPath-v0", 512, 1500, {}, 1000, "group_step_kernel<SAMPLED=1,G=16>"),
    _case("group32-TSP-N513", "TSP-v0", 513, 4000, {"parenting": 1}, 1000, "group_step_kernel<SAMPLED=1,G=32>"),
    _case("group32-Densest-N1024", "DensestSubgraph-v0", 1024, 3000, {"parenting": 1}, 1000, "group_step_kernel<SAMPLED=1,G=32>"),
    _case("tree-regs-Steiner-100-500", "SteinerTree-v0", 100, 500, {"n_dests": 5}, 1000, TREE % 8),                 # AW = 32 = 4 G
    _case("tree-walk-Multicast-p4-120-600", "MulticastRouting-v0", 120, 600, {"parenting": 4, "n_dests": 3}, 1000, TREE % 8),  # AW = 38
    _case("tree-chunks-Steiner-300-1200", "SteinerTree-v0", 300, 1200, {"n_dests": 5}, 1000, TREE % 16, chunks="chunks"),   # AW = 75: 15 + an empty chunk
    _case("tree-chunks-Multicast-p4-500-4000", "MulticastRouting-v0", 500, 4000, {"parenting": 4, "n_dests": 3}, 1000, TREE % 16,
          chunks="chunks"),                                                                                   # AW = 250: short last chunk
    _case("tree-chunks-Multicast-p3-600-2100", "MulticastRouting-v0", 600, 2100, {"parenting": 3, "n_dests": 3}, 1000, TREE % 32,
          chunks="chunks"),                                                                                   # AW = 132
    _case("tree-chunks-Steiner-1100-3000", "SteinerTree-v0", 1100, 3000, {"n_dests": 6}, 1000, TREE % 32, chunks="chunks"),  # NW = 35 > G
    _case("tree-regs-with-cnt-Multicast-p2-600-2000", "MulticastRouting-v0", 600, 2000, {"parenting": 2, "n_dests": 3}, 1000, TREE % 32,
          chunks="regs"),                                                                                     # AW = 125 <= 128
    _case("mis-N65", "MaxIndependentSet-v0", 65, 200, {}, 1000, MIS, T=70),
    _case("mis-N200", "MaxIndependentSet-v0", 200, 600, {}, 1000, MIS),
    _case("mis-N1100", "MaxIndependentSet-v0", 1100, 3000, {}, 1000, MIS),
    _case("dc-120-500", "DistributionCenter-v0", 120, 500, {"parenting": 2}, 1000, DC),
    _case("dc-500-4000", "DistributionCenter-v0", 500, 4000, {"parenting": 2, "target_count": 100, "max_distance": 1}, 1000, DC),
    _case("ppd-lane-N50", "PerishableProductDelivery-v0", 50, 200, {"n_products": 3, "parenting": 1}, 2900, "ppd_lane_step_kernel<SAMPLED=1>"),
    _case("ppd-lane-N64", "PerishableProductDelivery-v0", 64, 200, {"n_products": 3, "parenting": 1}, 2900, "ppd_lane_step_kernel<SAMPLED=1>"),
    _case("ppd-warp-N100", "PerishableProductDelivery-v0", 100, 300, {"n_products": 3, "parenting": 1}, 1000, "ppd_step_kernel<SAMPLED=1>"),
    _case("general-DistributionCenter-120-500", "DistributionCenter-v0", 120, 500, {"parenting": 2}, 1000, "step_kernel<SAMPLED=1,MINB=4>",
          force_warp=True),
]
SWEEP_ENV0 = 100003         # global env ids of a later rank
SWEEP_T0 = (1 << 32) - 23   # t + env_steps wraps at 2^32 after 23 steps
ORACLE_ENVS = 32
HOST_INSTANCES = 16         # N > 1024, beyond the device generator: host draws, repeated over the batch


def _sweep_batches(env_id, N, E, kw, B, force_warp):
    """Two identical batches (env_id0 = SWEEP_ENV0); the first keeps the env clock."""
    src = None
    if N > 1024:
        src = BatchedGraphEnv(env_id, HOST_INSTANCES, N, E, auto_reset=True, force_warp=force_warp, **kw)
        inst = []
        for b in range(HOST_INSTANCES):
            random.seed(1000 + b)
            np.random.seed(1000 + b)
            inst.append(generate_instance(env_id, src.params))
        src.load_instances(inst)
    envs = []
    for clock in (True, False):
        e = BatchedGraphEnv(env_id, B, N, E, auto_reset=True, env_id0=SWEEP_ENV0, force_warp=force_warp, **kw)
        if src is None:
            e.generate(seed=31)
        else:
            e.gather_instances(src, np.arange(B) % HOST_INSTANCES)
        e.reset()
        if clock:
            e.enable_env_clock()
        envs.append(e)
    return envs


@pytest.mark.parametrize("case", SWEEP)
def test_sampler_variant_draws_match_reference(case):
    """Every step of a short fused rollout: each env's drawn action against the reference, then the invariants; in lockstep
    a twin draws with ge_sample_actions and steps with ge_step, and the two end in the same state; an oracle slice
    replays the rollout.  The step's t starts 23 below 2^32, so t + env_steps wraps during the rollout."""
    env_id, N, E, kw, B, kernel, T, chunks, force_warp = case
    lo = B - ORACLE_ENVS - 5
    fz, tw = _sweep_batches(env_id, N, E, kw, B, force_warp)
    inst = fz.export_instances(lo, ORACLE_ENVS)
    assert fz.step_kernel_name(sampled=True) == kernel
    d = fz.desc
    G = 8 if d.NW <= 8 else 16 if d.NW <= 16 else 32
    assert ("mask_cnt" in fz.t) == (chunks is not None)
    if chunks == "chunks":
        assert d.AW > 4 * G and G >= 16, "group_sample_chunks draws only when AW > 4 G and G >= 16"
    elif chunks == "regs":
        assert d.AW <= 4 * G
    for k in range(T):
        tag = "%s step %d" % (kernel, k)
        fused_step_checked(fz, 7, SWEEP_T0, tag)
        tw.sample_actions(7, (SWEEP_T0 + k) & U32)
        tw.step_async(tw.actions_dev)
        assert_draws(tag + " vs ge_sample_actions", fz.actions_dev, tw.actions_dev.long(), fz.t["mask_bits"], None)
    torch.cuda.synchronize()
    check_invariants(tw, "twin")
    assert_same_state(fz, tw, kernel)
    oracle_slice_matches(fz, env_id, inst, lo, T, 7, SWEEP_T0 - (1 << 32), kernel)


def test_reference_draw_matches_oracle_sampler():
    """expected_draw == the oracle's oenv_sample_action row by row: empty, single-bit and full rows, rows whose only bits
    are bit 31 or bit 63, random densities, A not a multiple of 32, env clocks that make t + env_steps wrap."""
    rng = np.random.default_rng(5)
    for A in (32, 64, 75 * 32 - 7, 1000):
        AW = (A + 31) // 32
        rows = [np.zeros(A, bool), np.ones(A, bool)]
        for i in (0, 31, A - 1, min(63, A - 1)):
            r = np.zeros(A, bool)
            r[i] = True
            rows.append(r)
        rows += [rng.random(A) < p for p in (0.002, 0.01, 0.1, 0.5, 0.9, 0.99) for _ in range(12)]
        m = np.stack(rows)
        packed = np.zeros((m.shape[0], AW * 32), np.uint8)
        packed[:, :A] = m
        bits = torch.from_numpy(np.packbits(packed, axis=1, bitorder="little").view(np.int32).copy()).cuda()
        steps = rng.integers(0, 1 << 32, m.shape[0], dtype=np.uint64)
        steps[:8] = np.arange(8, dtype=np.uint64)
        for t, env0 in ((0, 0), (12345, 1 << 20), (U32 - 3, U32 - 40)):
            exp = expected_draw(bits, torch.from_numpy(steps.astype(np.int64)).cuda(), env0, 99, t).cpu().numpy()
            for b in range(m.shape[0]):
                want = orc.sample_action(m[b], 99, (env0 + b) & U32, (t + int(steps[b])) & U32)
                assert exp[b] == want, "A=%d row %d t=%d: reference %d, oracle %d" % (A, b, t, exp[b], want)
