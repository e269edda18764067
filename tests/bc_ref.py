"""Betweenness centrality as the tests restate it (include/essentials_b200.h, ess_bc), in float64 numpy.

brandes() follows the library's passes (BFS depths, σ forward over the levels, δ backward) over the edge list, so
parallel edges count as distinct paths and self-loops never lie on a shortest path. brute_force() is independent of
it: hop distances and path counts from every vertex, then δ_s(v) = Σ_t σ_sv σ_vt / σ_st wherever
d(s, v) + d(v, t) == d(s, t), straight from the definition."""
import numpy as np


def edge_list(off, col):
    off = np.asarray(off, np.int64)
    rows = np.repeat(np.arange(off.size - 1, dtype=np.int64), np.diff(off))
    return rows, np.asarray(col, np.int64)


def depths(n, rows, cols, s):
    """Hop distance from s over the edges rows -> cols; -1 = unreached."""
    depth = np.full(n, -1, np.int64)
    depth[s] = 0
    frontier = np.zeros(n, bool)
    frontier[s] = True
    d = 0
    while True:
        nxt = cols[frontier[rows]]
        nxt = np.unique(nxt[depth[nxt] < 0])
        if nxt.size == 0:
            return depth
        d += 1
        depth[nxt] = d
        frontier[:] = False
        frontier[nxt] = True


def dependencies(n, rows, cols, s):
    """(δ_s, depth) of one source, Brandes' recurrences over the levels."""
    depth = depths(n, rows, cols, s)
    sigma = np.zeros(n)
    sigma[s] = 1.0
    delta = np.zeros(n)
    deepest = int(depth.max())
    for d in range(1, deepest + 1):
        e = (depth[rows] == d - 1) & (depth[cols] == d)
        np.add.at(sigma, cols[e], sigma[rows[e]])
    for d in range(deepest - 1, -1, -1):
        e = (depth[rows] == d) & (depth[cols] == d + 1)
        u, w = rows[e], cols[e]
        np.add.at(delta, u, sigma[u] / sigma[w] * (1.0 + delta[w]))
    return delta, depth


def brandes(off, col, sources=None, scale=1.0):
    """bc[v] = scale · Σ_{s ∈ sources, s != v} δ_s(v) in float64; sources=None means every vertex."""
    n = len(off) - 1
    rows, cols = edge_list(off, col)
    acc = np.zeros(n)
    for s in range(n) if sources is None else sources:
        delta, _ = dependencies(n, rows, cols, int(s))
        delta[int(s)] = 0.0
        acc += delta
    return scale * acc


def brute_force(off, col, sources=None):
    """The same sum from the definition: all-pairs hop distances and path counts by plain BFS over adjacency lists."""
    n = len(off) - 1
    adj = [list(col[off[u]:off[u + 1]]) for u in range(n)]
    dist = np.full((n, n), -1, np.int64)
    paths = np.zeros((n, n))
    for a in range(n):
        dist[a, a], paths[a, a] = 0, 1.0
        queue = [a]
        for u in queue:
            for w in adj[u]:
                if dist[a, w] < 0:
                    dist[a, w] = dist[a, u] + 1
                    queue.append(w)
                if dist[a, w] == dist[a, u] + 1:
                    paths[a, w] += paths[a, u]
    bc = np.zeros(n)
    for s in range(n) if sources is None else sources:
        for v in range(n):
            if v == s or dist[s, v] < 0:
                continue
            for t in range(n):
                if t in (s, v) or dist[v, t] < 0 or dist[s, t] != dist[s, v] + dist[v, t]:
                    continue
                bc[v] += paths[s, v] * paths[v, t] / paths[s, t]
    return bc


def from_edges(n, src, dst):
    """CSR (int64 offsets, int32 columns, rows in (src, dst) order) of a directed multigraph."""
    src, dst = np.asarray(src, np.int64), np.asarray(dst, np.int64)
    order = np.lexsort((dst, src))
    off = np.zeros(n + 1, np.int64)
    np.add.at(off, src + 1, 1)
    return np.cumsum(off), dst[order].astype(np.int32)


def random_multigraph(rng, symmetric):
    """Small graph with self-loops, parallel edges, isolated vertices and (usually) several components."""
    n = int(rng.integers(2, 28))
    m = int(rng.integers(1, 3 * n))
    src, dst = rng.integers(0, n, m), rng.integers(0, n, m)
    dup = rng.integers(0, m, m // 4 + 1)  # parallel edges
    src, dst = np.concatenate([src, src[dup]]), np.concatenate([dst, dst[dup]])
    if symmetric:
        src, dst = np.concatenate([src, dst]), np.concatenate([dst, src])
    return n, src, dst
