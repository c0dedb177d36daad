"""GPU: the structural-feature kernels (csrc/ge_features.cu) at every dispatch branch against the C oracle's fp64 values
(oracle/graphenvs_oracle.c:oenv_features, itself pinned to networkx by test_features_reference.py).

Contract, per node and column, against np.float32(oracle):
  * degree, closeness, clustering: bit-identical (integer counts and the same fp64 expression on both sides);
  * betweenness, pagerank: within 1 float32 ulp, and exactly 0 where the oracle gives 0 (the sums are reassociated, so the
    fp64 values differ by ~1e-15 relative and may round to neighbouring floats).
Every shape runs through the dispatch ge_features picks and through the warp-per-env family (force_warp), and the kernel
actually launched is read back from a CUDA activity trace and compared with `_features_launch`."""
import json
import random
import re
import time

import numpy as np
import pytest
import torch

import cuda_util as cu
import feature_graphs as fg
from graphenvs_b200 import BatchedGraphEnv
from graphenvs_b200.instances import Instance, generate_instance
from graphenvs_b200.spec import check_ctor_args

pytestmark = pytest.mark.gpu

MIS, TSP = "MaxIndependentSet-v0", "TSP-v0"
GE_WPB = 8   # warps (= envs) per block of the warp family, csrc/ge_common.cuh


# ---------------------------------------------------------------------------------------------------- dispatch mirror
def _feat_nwp(NW):
    q = (NW + 3) >> 2
    return (q + 1 - (q & 1)) << 2


def _features_launch(N, M, force_warp=False, B=1):
    """The kernel ge_features launches for a batch of shape (N, M), restated from its host code
    (csrc/ge_features.cu:ge_features, lines 569-606, and launch_warp_family, lines 552-565)."""
    NW = (N + 31) // 32
    budget = 227 * 1024
    cta_fits = True
    if N <= 1024 and not force_warp:
        NWP = _feat_nwp(NW)
        wb = (16 * N + 4 * NWP + 2 * N + 15) & ~15                    # sigma | delta | level set | D, per warp
        mat = N * NWP * 4
        avg = M // N
        csrp = avg <= 32 and M < 65536
        csr_bytes = ((2 * (N + 1) + 2 * M + 15) & ~15) if csrp else 0
        dropped = csrp and mat + csr_bytes + 4 * wb + 128 > budget
        if dropped:
            csrp, csr_bytes = False, 0
        W = min(max((N + 7) // 8, 2), 16)
        while W > 2 and mat + csr_bytes + W * wb + 128 > budget:
            W -= 1
        smem = mat + csr_bytes + max(W * wb + 128, 3 * N * 8 + 128)
        cta_fits = smem <= budget
        if cta_fits:
            G = 1
            while G < 32 and 2 * G <= avg // 2:
                G <<= 1
            nwmax = next(k for k in (2, 4, 8, 16, 32) if NW <= k)
            return dict(family="cta", NWMAX=nwmax, CSRP=csrp, W=W, G=G, dropped=dropped,
                        grid=[B, 1, 1], block=[32 * W, 1, 1])
    words = (7 * N + 3 * NW + 3) & ~3                                  # feat_words: sigma, delta, bt, D, 3 bitsets
    wpb = min((200 * 1024) // (4 * words), GE_WPB)
    return dict(family="warp", wpb=wpb, fallback=not cta_fits, grid=[(B + wpb - 1) // wpb, 1, 1], block=[32 * wpb, 1, 1])


def _launched(ev):
    """(family, NWMAX, CSRP, grid, block) of a features kernel's trace event."""
    name, args = ev["name"], ev["args"]
    m = re.search(r"features_cta_kernel<(\d+), (true|false)>", name) or re.search(r"features_cta_kernelILi(\d+)ELb([01])E", name)
    if m:
        return "cta", int(m.group(1)), m.group(2) in ("true", "1"), args["grid"], args["block"]
    assert "features_warp_kernel" in name, name
    return "warp", None, None, args["grid"], args["block"]


# ---------------------------------------------------------------------------------------------------- the shapes
def _family(env_id, n, e, builder, relabel=True):
    """Instance b: builder(rng) with node ids permuted for b >= 1 (env 0 keeps the canonical labels, whose level sets
    are contiguous bit runs); TSP carries non-uniform symmetric weights (weighted pagerank)."""
    def make(b):
        rng = np.random.default_rng(7000 + b)
        edges = builder(rng)
        if relabel and b >= 1:
            edges = fg.relabel(edges, n, rng)
        assert len(edges) == e
        w = fg.nonuniform_weights(len(edges), rng) if env_id == TSP else None
        links, w64 = fg.links(n, edges, rng, w)
        return Instance(n_nodes=n, links=links, w64=w64, node_cost=np.zeros(n) if env_id == MIS else None)
    return make


def _draw(env_id, n, e, kw):
    """The reference's own seeded instance (generate_instance), in its own kind."""
    p = check_ctor_args(env_id, n, e, dict(kw))

    def make(b):
        random.seed(60 + b)
        np.random.seed(60 + b)
        return generate_instance(env_id, p)
    return make


def _case(name, env_id, n, e, B, make, kw=None):
    kw = dict(kw or ({"parenting": 1} if env_id == TSP else {}))
    return pytest.param((env_id, n, e, B, make, kw), id=name)


# Unweighted graphs load into MaxIndependentSet-v0, weighted ones into TSP-v0: both are node-action kinds (edge-action
# kinds refuse degree-0 nodes) and their loading runs no search that would reject an arbitrary graph.  The expected
# dispatch in the comments is what _features_launch gives (CSR = the 16-bit CSR gathers, dense = the bit-word loops).
CASES = [
    _case("tsp_complete_40", TSP, 40, 780, 3, _family(TSP, 40, 780, lambda r: fg.complete(40))),              # <2,dense> W5 G16
    _case("tsp_complete_64", TSP, 64, 2016, 3, _family(TSP, 64, 2016, lambda r: fg.complete(64))),            # <2,dense> W8 G16
    _case("complete_20", MIS, 20, 190, 3, _family(MIS, 20, 190, lambda r: fg.complete(20))),                  # <2,CSR> W3 G8
    _case("gnm_100_2000", MIS, 100, 2000, 3, _family(MIS, 100, 2000, lambda r: fg.gnm(100, 2000, r))),        # <4,dense> W13
    _case("tsp_gnm_100_300", TSP, 100, 300, 3, _family(TSP, 100, 300, lambda r: fg.gnm(100, 300, r))),        # <4,CSR> G2, weighted
    _case("tsp_complete_128", TSP, 128, 8128, 2, _family(TSP, 128, 8128, lambda r: fg.complete(128))),        # <4,dense> W16 G32
    _case("gnm_250_5000", MIS, 250, 5000, 3, _family(MIS, 250, 5000, lambda r: fg.gnm(250, 5000, r))),        # <8,dense>
    _case("gnm_256_1000", MIS, 256, 1000, 3, _family(MIS, 256, 1000, lambda r: fg.gnm(256, 1000, r))),        # <8,CSR>
    _case("gnm_400_8000", MIS, 400, 8000, 3, _family(MIS, 400, 8000, lambda r: fg.gnm(400, 8000, r))),        # <16,dense>
    _case("tsp_complete_512", TSP, 512, 130816, 2, _family(TSP, 512, 130816, lambda r: fg.complete(512))),    # <16,dense> G32
    _case("ring_of_cliques_20x35", MIS, 700, 11920, 3,                                                        # <32,dense> W12,
          _family(MIS, 700, 11920, lambda r: fg.ring_of_cliques(20, 35))),                                    # ~20 levels
    _case("gnm_1000_5000", MIS, 1000, 5000, 3, _family(MIS, 1000, 5000, lambda r: fg.gnm(1000, 5000, r))),    # <32,dense> W4,
    #                                                                                               CSR dropped by budget
    _case("tsp_complete_1024", TSP, 1024, 523776, 2, _family(TSP, 1024, 523776, lambda r: fg.complete(1024))),  # <32,dense>
    _case("path_1024", MIS, 1024, 1023, 3, _family(MIS, 1024, 1023, lambda r: fg.path(1024))),                # <32,CSR> W4 G1,
    _case("cycle_1024", MIS, 1024, 1024, 3, _family(MIS, 1024, 1024, lambda r: fg.cycle(1024))),              # 1023 / 512 levels
    _case("grid_32x32", MIS, 1024, 1984, 3, _family(MIS, 1024, 1984, lambda r: fg.grid(32, 32))),             # C(62,31) > 2^53
    _case("star_1024", MIS, 1024, 1023, 2, _family(MIS, 1024, 1023, lambda r: fg.star(1024))),                # centre: exactly 1
    _case("components_300", MIS, 300, 539, 3, _family(MIS, 300, 539, lambda r: fg.components(300, r))),      # <16,CSR>
    _case("n2_edge", MIS, 2, 1, 3, _family(MIS, 2, 1, lambda r: fg.path(2))),                                 # <2,CSR> W2,
    _case("n2_edgeless", MIS, 2, 0, 3, _family(MIS, 2, 0, lambda r: fg.path(1))),                             # _rescale's
    _case("n3_path", MIS, 3, 2, 3, _family(MIS, 3, 2, lambda r: fg.path(3))),                                 # N <= 2 branch
    _case("n3_one_edge", MIS, 3, 1, 3, _family(MIS, 3, 1, lambda r: fg.path(2))),
    _case("tsp_triangle", TSP, 3, 3, 3, _family(TSP, 3, 3, lambda r: fg.complete(3))),
    _case("gnm_1025_3000", MIS, 1025, 3000, 3, _family(MIS, 1025, 3000, lambda r: fg.gnm(1025, 3000, r))),   # warp family
    _case("gnm_1100_55000", MIS, 1100, 55000, 2, _family(MIS, 1100, 55000, lambda r: fg.gnm(1100, 55000, r))),
    _case("gnm_4096_8192", MIS, 4096, 8192, 2, _family(MIS, 4096, 8192, lambda r: fg.gnm(4096, 8192, r))),   # 1 warp/block
    # the reference's own seeded draws at the CTA instantiations the golden fixtures do not reach
    _case("draw_tsp_40_780", TSP, 40, 780, 3, _draw(TSP, 40, 780, {"parenting": 1})),                         # <2,dense>
    _case("draw_longest_100_2000", "LongestPath-v0", 100, 2000, 3,                                           # <4,dense>
          _draw("LongestPath-v0", 100, 2000, {"parenting": 1}), {"parenting": 1}),
    _case("draw_densest_400_8000", "DensestSubgraph-v0", 400, 8000, 3,                                       # <16,dense>
          _draw("DensestSubgraph-v0", 400, 8000, {"parenting": 1}), {"parenting": 1}),
    _case("draw_shortest_1000_5000", "ShortestPath-v0", 1000, 5000, 3,                                       # CSR dropped
          _draw("ShortestPath-v0", 1000, 5000, {})),
    _case("draw_tsp_800_16000", TSP, 800, 16000, 2, _draw(TSP, 800, 16000, {"parenting": 1})),                # <32,dense>
    _case("draw_tsp_700_6000", TSP, 700, 6000, 2, _draw(TSP, 700, 6000, {"parenting": 1})),                   # <32,CSR> G8
]


# ---------------------------------------------------------------------------------------------------- helpers
def _ordered(x):
    """float32 -> integers in the order of the floats: adjacent floats differ by 1."""
    i = np.ascontiguousarray(x, dtype=np.float32).view(np.int32).astype(np.int64)
    return np.where(i < 0, -(i & 0x7fffffff), i)


def _assert_contract(got, ref64, tag):
    ref = ref64.astype(np.float32)
    for c, what in ((0, "degree"), (2, "closeness"), (4, "clustering")):
        bad = np.flatnonzero(got[:, c].view(np.int32) != ref[:, c].view(np.int32))
        assert bad.size == 0, "%s %s not bit-identical at nodes %s: got %r, oracle %r" % (
            tag, what, bad[:5], got[bad[:5], c], ref64[bad[:5], c])
    for c, what in ((1, "betweenness"), (3, "pagerank")):
        zero = ref64[:, c] == 0.0
        bad = np.flatnonzero(zero & (got[:, c] != 0.0))
        assert bad.size == 0, "%s %s nonzero where the oracle gives 0, nodes %s: %r" % (tag, what, bad[:5], got[bad[:5], c])
        ulps = np.abs(_ordered(got[:, c]) - _ordered(ref[:, c]))
        bad = np.flatnonzero(ulps > 1)
        assert bad.size == 0, "%s %s off by %d float32 ulps at nodes %s: got %r, oracle %r" % (
            tag, what, ulps.max(), bad[:5], got[bad[:5], c], ref64[bad[:5], c])


def _batch(env_id, instances, kw, force_warp):
    """A batch with the instances loaded and no features computed yet."""
    ins = instances[0]
    env = BatchedGraphEnv(env_id, len(instances), ins.n_nodes, len(ins.links) // 2, force_warp=force_warp, **kw)
    env.load_instances(instances)
    return env


def _oracle(env_id, ins, params):
    return cu.oracle_from_instance(env_id, ins, params).features64(weighted_pr=(env_id == TSP))


# ---------------------------------------------------------------------------------------------------- tests
def test_launched_kernel_matches_mirror(tmp_path):
    """For every shape of the table, the kernel compute_features() launches (name, grid, block) read back from a CUDA
    activity trace equals _features_launch's: the default dispatch everywhere, force_warp where the warp family is cheap.

    All launches go into one trace, opened and closed with a second of margin and taken first thing in the module: with
    one short trace per launch, the kernel record was missing from about half of the traces taken after the first 20 s
    of a B200 run (the launch itself was recorded)."""
    from torch.profiler import ProfilerActivity, profile
    launches = []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        time.sleep(1.0)
        for p in CASES:
            env_id, n, e, B, make, kw = p.values[0]
            for fw in (False, True) if n <= 300 else (False,):
                env = _batch(env_id, [make(b) for b in range(B)], kw, fw)
                env.compute_features()
                torch.cuda.synchronize()
                launches.append(("%s force_warp=%s" % (p.id, fw), _features_launch(n, 2 * e, fw, B)))
                del env
        time.sleep(1.0)
    path = tmp_path / "features_trace.json"
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    ks = sorted((ev for ev in events if ev.get("cat") == "kernel" and "features_" in ev.get("name", "")), key=lambda ev: ev["ts"])
    assert len(ks) == len(launches), ("features kernels traced:", [ev["name"] for ev in ks], len(launches))
    for (tag, want), ev in zip(launches, ks):
        family, nwmax, csrp, grid, block = _launched(ev)
        assert family == want["family"], (tag, ev["name"], want)
        if family == "cta":
            assert (nwmax, csrp) == (want["NWMAX"], want["CSRP"]), (tag, ev["name"], want)
        assert list(grid) == want["grid"] and list(block) == want["block"], (tag, grid, block, want)


@pytest.mark.parametrize("case", CASES)
def test_features_match_oracle_at_every_dispatch(case):
    """Both families, every shape: the features meet the contract against the oracle.  The CTA kernel has no
    floating-point atomics: a second call is bit-identical."""
    env_id, n, e, B, make, kw = case
    instances = [make(b) for b in range(B)]
    params = check_ctor_args(env_id, n, e, dict(kw))
    ref = [_oracle(env_id, ins, params) for ins in instances]
    for force_warp in (False, True):
        env = _batch(env_id, instances, kw, force_warp)
        feats = env.compute_features().cpu().numpy().copy()
        family = _features_launch(n, 2 * e, force_warp)["family"]
        tag = "%s %s" % (env_id, family)
        for b in range(B):
            _assert_contract(feats[b], ref[b], "%s env %d" % (tag, b))
        if family == "cta":
            again = env.compute_features().cpu().numpy()
            assert np.array_equal(again.view(np.int32), feats.view(np.int32)), tag + ": second call differs"


def test_dispatch_coverage():
    """The table above reaches every instantiation and every budget decision of ge_features.  The first test checks from
    the trace that the launched kernel is the mirror's, so these are launches, not assumptions."""
    seen = []
    for p in CASES:
        env_id, n, e, B, make, kw = p.values[0]
        for fw in (False, True):
            d = _features_launch(n, 2 * e, fw, B)
            d["weighted"] = env_id == TSP
            seen.append(d)
    cta = [d for d in seen if d["family"] == "cta"]
    pairs = {(d["NWMAX"], d["CSRP"]) for d in cta}
    assert pairs == {(k, c) for k in (2, 4, 8, 16, 32) for c in (False, True)}, sorted(pairs)
    assert any(d["family"] == "warp" for d in seen)
    assert any(d["family"] == "warp" and d["wpb"] == 1 for d in seen)      # N = 4096: one warp per block
    Ws = {d["W"] for d in cta}
    assert {2, 3, 4, 16} <= Ws and any(4 < w < 16 for w in Ws), sorted(Ws)
    assert {1, 2, 4, 8, 16, 32} <= {d["G"] for d in cta}, sorted({d["G"] for d in cta})
    assert any(d["dropped"] for d in cta)
    assert any(d["weighted"] and d["CSRP"] for d in cta) and any(d["weighted"] and not d["CSRP"] for d in cta)


def _mixed_batches():
    """(env_id, kw, 5 instances of one (N, M), the instance of interest = index 3)."""
    r = np.random.default_rng(11)

    def mis(n, edges):
        links, w64 = fg.links(n, edges, r)
        return Instance(n_nodes=n, links=links, w64=w64, node_cost=np.zeros(n))
    yield "path_in_trees", MIS, {}, [mis(1024, fg.star(1024)), mis(1024, fg.gnm(1024, 1023, r)), mis(1024, fg.gnm(1024, 1023, r)),
                                     mis(1024, fg.relabel(fg.path(1024), 1024, r)), mis(1024, fg.relabel(fg.star(1024), 1024, r))]
    yield "gnm_1000_5000", MIS, {}, [mis(1000, fg.gnm(1000, 5000, r)) for _ in range(5)]
    yield "ring_in_gnm", MIS, {}, [mis(700, fg.gnm(700, 11920, r)) for _ in range(3)] + [
        mis(700, fg.relabel(fg.ring_of_cliques(20, 35), 700, r)), mis(700, fg.gnm(700, 11920, r))]
    yield "tsp_gnm_100_2000", TSP, {"parenting": 1}, [_draw(TSP, 100, 2000, {"parenting": 1})(b) for b in range(5)]
    yield "gnm_1100_3000", MIS, {}, [mis(1100, fg.gnm(1100, 3000, r)) for _ in range(5)]


@pytest.mark.parametrize("name", ["path_in_trees", "gnm_1000_5000", "ring_in_gnm", "tsp_gnm_100_2000", "gnm_1100_3000"])
def test_features_independent_of_batch_position(name):
    """An env's features do not depend on its index or on the other envs of the batch: B = 1 equals index 3 of a mixed
    batch of other graphs of the same (N, M).  Bit-identical for the CTA kernel; the warp family adds delta with fp64
    atomics, whose order is not fixed, so it is held to the ulp contract against the oracle instead."""
    _, env_id, kw, inst = next(m for m in _mixed_batches() if m[0] == name)
    n, e = inst[0].n_nodes, len(inst[0].links) // 2
    alone = _batch(env_id, [inst[3]], kw, False).compute_features().cpu().numpy()[0]
    mixed = _batch(env_id, inst, kw, False).compute_features().cpu().numpy()[3]
    if _features_launch(n, 2 * e)["family"] == "cta":
        assert np.array_equal(alone.view(np.int32), mixed.view(np.int32)), name
    else:
        ref = _oracle(env_id, inst[3], check_ctor_args(env_id, n, e, dict(kw)))
        _assert_contract(alone, ref, name + " alone")
        _assert_contract(mixed, ref, name + " at index 3")


@pytest.mark.parametrize("cfg", [("TSP-v0", 40, 780, {"parenting": 1}), ("DensestSubgraph-v0", 400, 8000, {"parenting": 1}),
                                 ("ShortestPath-v0", 1100, 3000, {})], ids=lambda c: "%s-N%d" % (c[0][:-3], c[1]))
def test_obs_wire_format_with_features(cfg):
    """obs_flat() with structural features on == the oracle's obs() built with the device's features, at reset and over a
    few random valid steps (the feature columns sit between the dynamic node columns and the edge block)."""
    env_id, n, e, kw = cfg
    B, seed = 3, 5
    env = BatchedGraphEnv(env_id, B, n, e, auto_reset=True, structural_features=True, **kw)
    inst = [_draw(env_id, n, e, kw)(b) for b in range(B)]
    env.load_instances(inst)
    env.reset()
    feats = env.t["features"].cpu().numpy()
    assert np.all(feats[:, :, 3] > 0)   # pagerank: the features are there
    oenvs = [cu.oracle_from_instance(env_id, i, env.params, features=feats[b]) for b, i in enumerate(inst)]
    for t in range(4):
        obs = env.obs_flat().cpu().numpy()
        for b, oe in enumerate(oenvs):
            np.testing.assert_array_equal(obs[b], oe.obs(), err_msg="obs env %d after %d steps" % (b, t))
        acts = env.sample_actions(seed, t).cpu().numpy()
        env.step(env.actions_dev)
        torch.cuda.synchronize()
        for b, oe in enumerate(oenvs):
            if oe.step(int(acts[b]))["done"]:
                oe.reset_state()
