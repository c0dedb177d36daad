"""Graph families for the structural-feature tests (test_cuda_features.py, test_features_reference.py).

Each builder returns the undirected edges of a simple graph as int64 [E, 2].  `links()` turns them into the
reference's link order: both directions of every edge, rows in ascending source order, each row in a shuffled
neighbour order (the reference's rows follow insertion order, not neighbour id), with symmetric weights."""
import numpy as np


def complete(n):
    return np.stack(np.triu_indices(n, 1), 1).astype(np.int64)


def path(n):
    a = np.arange(n - 1, dtype=np.int64)
    return np.stack([a, a + 1], 1)


def cycle(n):
    return np.concatenate([path(n), [[n - 1, 0]]]).astype(np.int64)


def star(n):
    a = np.arange(1, n, dtype=np.int64)
    return np.stack([np.zeros_like(a), a], 1)


def grid(r, c):
    """r x c lattice: the corner-to-corner shortest-path count is C(r+c-2, r-1)."""
    ids = np.arange(r * c, dtype=np.int64).reshape(r, c)
    return np.concatenate([np.stack([ids[:, :-1].ravel(), ids[:, 1:].ravel()], 1),
                           np.stack([ids[:-1, :].ravel(), ids[1:, :].ravel()], 1)])


def ring_of_cliques(k, c):
    """k cliques of c nodes; the last node of clique i is joined to the first node of clique i+1 (mod k), so a search
    crosses each clique in two levels."""
    e = [complete(c) + i * c for i in range(k)]
    e.append(np.array([[i * c + c - 1, ((i + 1) % k) * c] for i in range(k)], dtype=np.int64))
    return np.concatenate(e)


def gnm(n, m, rng):
    """m distinct uniformly drawn edges on n nodes (not necessarily connected)."""
    assert m <= n * (n - 1) // 2
    codes = np.zeros(0, np.int64)
    while codes.size < m:
        u = rng.integers(0, n, 2 * m)
        v = rng.integers(0, n, 2 * m)
        keep = u != v
        lo, hi = np.minimum(u, v)[keep], np.maximum(u, v)[keep]
        new = lo * n + hi
        _, first = np.unique(np.concatenate([codes, new]), return_index=True)
        codes = np.concatenate([codes, new])[np.sort(first)]
    codes = codes[:m]
    return np.stack([codes // n, codes % n], 1)


def components(n, rng):
    """Two components of unequal size and diameter plus isolated nodes: a G(n, m) draw on the first 40 % of the nodes,
    a path with a chord every 11 nodes on the next 55 %, the rest isolated (closeness over fewer than n reached nodes,
    dangling pagerank mass).  The edge count depends on n only."""
    a, b = int(0.4 * n), int(0.55 * n)
    ea = gnm(a, 3 * a, rng)
    eb = path(b) + a
    lo = np.arange(a, a + b - 7, 11, dtype=np.int64)
    return np.concatenate([ea, eb, np.stack([lo, lo + 7], 1)])


def relabel(edges, n, rng):
    """The same graph under a random permutation of the node ids."""
    return rng.permutation(n)[np.asarray(edges, np.int64)]


def links(n, edges, rng, weights=None):
    """(links int32 [2E, 2], w64 float64 [2E]) in the reference's order.  `weights` is one value per undirected edge
    (both directions carry it); None -> 1.0."""
    e = np.asarray(edges, np.int64).reshape(-1, 2)
    d = np.concatenate([e, e[:, ::-1]])
    w = np.ones(len(e)) if weights is None else np.asarray(weights, np.float64)
    w = np.concatenate([w, w])
    order = np.lexsort((rng.permutation(len(d)), d[:, 0]))
    assert n > 0 and (d.size == 0 or d.max() < n)
    return d[order].astype(np.int32), w[order]


def nonuniform_weights(n_edges, rng):
    """Symmetric edge weights for weighted pagerank, spread over a decade so that row sums differ."""
    return rng.uniform(0.1, 1.0, n_edges)
