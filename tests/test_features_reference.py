"""CPU: the C oracle's structural features (oracle/graphenvs_oracle.c:oenv_features) against networkx on the graph
families of test_cuda_features.py, at the sizes where networkx's Python Brandes runs in seconds (N * M <= ~2e7).  With
that file (device == oracle to the float32 ulp) this chains device -> oracle -> networkx for every family, including the
sizes networkx is too slow for.

The networkx side restates oracle/gen_golden.py:nx_features64 on the graph the reference hands to
feature_extraction.generate_features: a DiGraph with nodes 0..N-1 and the links in reference order, the edge weight
under 'weight' only for TSP (the attribute nx.pagerank reads; the other kinds store 'delay', so their pagerank is
unweighted)."""
import numpy as np
import pytest

import feature_graphs as fg
from oracle import oracle as orc

nx = pytest.importorskip("networkx", reason="networkx is the reference's feature library; without it there is nothing to pin the oracle to")

FAMILIES = {
    "complete_20": (20, lambda r: fg.complete(20)),
    "complete_40_weighted": (40, lambda r: fg.complete(40)),
    "complete_128_weighted": (128, lambda r: fg.complete(128)),
    "gnm_100_2000": (100, lambda r: fg.gnm(100, 2000, r)),
    "gnm_100_300_weighted": (100, lambda r: fg.gnm(100, 300, r)),
    "gnm_400_8000": (400, lambda r: fg.gnm(400, 8000, r)),
    "gnm_1000_5000": (1000, lambda r: fg.gnm(1000, 5000, r)),
    "gnm_1025_3000": (1025, lambda r: fg.gnm(1025, 3000, r)),
    "ring_of_cliques_12x12": (144, lambda r: fg.ring_of_cliques(12, 12)),
    "path_1024": (1024, lambda r: fg.path(1024)),
    "cycle_1024": (1024, lambda r: fg.cycle(1024)),
    "grid_32x32": (1024, lambda r: fg.grid(32, 32)),
    "star_1024": (1024, lambda r: fg.star(1024)),
    "components_300": (300, lambda r: fg.components(300, r)),
    "components_300_weighted": (300, lambda r: fg.components(300, r)),
    "n2_edge": (2, lambda r: fg.path(2)),
    "n2_edgeless": (2, lambda r: fg.path(1)),
    "n3_path": (3, lambda r: fg.path(3)),
    "n3_one_edge": (3, lambda r: fg.path(2)),
    "triangle_weighted": (3, lambda r: fg.complete(3)),
}


def nx_features64(n, links, w64, weighted):
    G = nx.DiGraph()
    G.add_nodes_from(range(n))
    for (u, v), w in zip(links.tolist(), w64.tolist()):
        if weighted:
            G.add_edge(u, v, weight=w)
        else:
            G.add_edge(u, v)
    cl = nx.clustering(G)
    pr = nx.pagerank(G)
    bt = nx.betweenness_centrality(G)
    cs = nx.closeness_centrality(G)
    return np.array([[G.degree(v), bt[v], cs[v], pr[v], cl[v]] for v in G.nodes], dtype=np.float64)


@pytest.mark.parametrize("name", list(FAMILIES))
def test_oracle_features_match_networkx(name):
    n, build = FAMILIES[name]
    weighted = name.endswith("weighted")
    rng = np.random.default_rng(3)
    edges = fg.relabel(build(rng), n, rng)
    links, w64 = fg.links(n, edges, rng, fg.nonuniform_weights(len(edges), rng) if weighted else None)
    kind = orc.KINDS["TSP-v0" if weighted else "ShortestPath-v0"]
    got = orc.OracleEnv(kind, n, links, w64).features64(weighted_pr=weighted)
    want = nx_features64(n, links, w64, weighted)
    np.testing.assert_array_equal(got[:, 0], want[:, 0])
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=0, err_msg=name)
