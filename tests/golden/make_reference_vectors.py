"""Generates tests/golden/reference_outputs.npz: what the reference's own code returns on the inputs of the tests that
compare with it (tests/test_oracle.py, tests/test_io.py, tests/test_gpu_vs_reference_gpu.py), so that those
comparisons also run where the reference's build (oracle/_ref) is absent.   python tests/golden/make_reference_vectors.py

Only outputs with exactly one right answer are stored, and each is computed here by a small NumPy implementation that
shares no code with the oracle or the CUDA path, then cross-checked against the oracle:
 - BFS depths (unreached = 2^31 - 1, as the reference's bfs_cpu and bfs::run report them);
 - SSSP distances in float32: the least fixed point of d[v] = min(d[v], fl32(d[u] + w)) with d[source] = 0, which the
   reference's sssp_cpu (Dijkstra) and its GPU sssp::run (atomic-min relaxation) both reach bit for bit
   (unreached = FLT_MAX);
 - k-core numbers (peeling, every CSR entry counts towards the degree).
PageRank, PPR, colouring and the reference's random stream have no unique answer and are not stored.
The `.csr` files are what essentials_b200.io.write_csr_binary writes for test_io's graphs; that writer has not
changed since it was checked byte for byte against the reference's csr_t::write_binary.
"""
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from essentials_b200 import graphgen as gg  # noqa: E402
from essentials_b200 import io as eio  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_outputs.npz")
INF = 2**31 - 1
FLT_MAX = np.float32(3.4028234663852886e38)


def _rows(off):
    return np.repeat(np.arange(off.size - 1), np.diff(off))


def bfs(off, col, s):
    off, col = off.astype(np.int64), col.astype(np.int64)
    rows = _rows(off)
    d = np.full(off.size - 1, INF, np.int64)
    d[s] = 0
    level = 0
    while True:
        nxt = col[d[rows] == level]
        nxt = np.unique(nxt[d[nxt] == INF])
        if nxt.size == 0:
            return d.astype(np.int32)
        level += 1
        d[nxt] = level


def sssp(off, col, w, s):
    rows = _rows(off.astype(np.int64))
    col = col.astype(np.int64)
    w = w.astype(np.float32)
    d = np.full(off.size - 1, np.inf, np.float32)
    d[s] = 0
    while True:
        via = d[rows] + w  # float32 + float32: one rounding, as in C
        new = d.copy()
        np.minimum.at(new, col, via)
        if np.array_equal(new, d):
            return np.where(np.isinf(d), FLT_MAX, d).astype(np.float32)
        d = new


def kcore(off, col):
    n = off.size - 1
    deg = np.diff(off).astype(np.int64)
    core = np.zeros(n, np.int32)
    removed = np.zeros(n, bool)
    k = 0
    while not removed.all():
        k = max(k, int(deg[~removed].min()))
        while True:
            peel = np.flatnonzero(~removed & (deg <= k))
            if peel.size == 0:
                break
            core[peel] = k
            removed[peel] = True
            for v in peel:
                np.subtract.at(deg, col[off[v]:off[v + 1]], 1)
    return core


def small_multigraphs(count=120, seed=7):
    """Fixed directed multigraphs like the property test draws: self loops, parallel edges, isolated and unreachable
    vertices, zero and repeated dyadic weights."""
    rng = np.random.default_rng(seed)
    weights = np.array([0.0, 0.5, 1.0, 1.0, 2.25, 7.0, 63.984375], np.float32)
    for _ in range(count):
        n = int(rng.integers(1, 25))
        m = int(rng.integers(0, 81))
        src, dst = rng.integers(0, n, m), rng.integers(0, n, m)
        w = weights[rng.integers(0, weights.size, m)]
        order = np.lexsort((dst, src))
        off = np.zeros(n + 1, np.int64)
        np.add.at(off, src + 1, 1)
        yield np.cumsum(off), dst[order].astype(np.int32), w[order], int(rng.integers(0, n))


def main():
    d = {}

    def put_paths(prefix, off, col, val, sources):
        d[f"{prefix}_sources"] = np.array(sources, np.int32)
        for s in sources:
            d[f"{prefix}_bfs_{s}"] = bfs(off, col, s)
            assert np.array_equal(d[f"{prefix}_bfs_{s}"], oracle.bfs(off, col, s)), (prefix, s)
            if val is not None:
                d[f"{prefix}_sssp_{s}"] = sssp(off, col, val, s)
                assert np.array_equal(d[f"{prefix}_sssp_{s}"], oracle.sssp(off, col, val, s)), (prefix, s)

    # tests/test_oracle.py::test_oracle_matches_reference_code_on_fresh_graphs
    for scale, seed in ((8, 3), (11, 5), (12, 1)):
        g = gg.rmat_csr(scale, seed=seed, weights="hash")
        off, col, val = g.host()
        put_paths(f"rmat{scale}", off, col, val, gg.pick_sources(g, 2, seed=seed))
        d[f"rmat{scale}_kcore"] = kcore(off, col)
        assert np.array_equal(d[f"rmat{scale}_kcore"], oracle.kcore(off, col)), scale
    off, col, val = gg.grid_csr(40, 31).host()
    d["grid40x31_sssp_5"] = sssp(off, col, val, 5)
    assert np.array_equal(d["grid40x31_sssp_5"], oracle.sssp(off, col, val, 5))
    # ...::test_oracle_matches_reference_code_on_arbitrary_small_graphs
    for i, (off, col, w, s) in enumerate(small_multigraphs()):
        d[f"mg{i}_offsets"], d[f"mg{i}_indices"], d[f"mg{i}_values"], d[f"mg{i}_source"] = off, col, w, np.int32(s)
        d[f"mg{i}_bfs"], d[f"mg{i}_sssp"] = bfs(off, col, s), sssp(off, col, w, s)
        assert np.array_equal(d[f"mg{i}_bfs"], oracle.bfs(off, col, s)), i
        assert np.array_equal(d[f"mg{i}_sssp"], oracle.sssp(off, col, w, s)), i
    # tests/test_gpu_vs_reference_gpu.py: BFS and SSSP on Kronecker scale 15, k-core on scale 11
    g = gg.rmat_csr(15, weights="hash")
    off, col, val = g.host()
    put_paths("kron15", off, col, None, [0] + gg.pick_sources(g, 2))
    s = gg.pick_sources(g, 1)[0]
    d["kron15_sssp_source"] = np.int32(s)
    d[f"kron15_sssp_{s}"] = sssp(off, col, val, s)
    assert np.array_equal(d[f"kron15_sssp_{s}"], oracle.sssp(off, col, val, s))
    off, col, _ = gg.rmat_csr(11).host()
    d["kron11_kcore"] = kcore(off, col)
    assert np.array_equal(d["kron11_kcore"], oracle.kcore(off, col))
    # tests/test_io.py: the .csr files of its three graphs
    with tempfile.TemporaryDirectory() as tmp:
        for i, csr in enumerate((gg.rmat_csr(8, weights="hash"), gg.grid_csr(7, 5),
                                 gg.rmat_csr(6, symmetric=False, weights="none"))):
            path = os.path.join(tmp, f"{i}.csr")
            eio.write_csr_binary(path, csr)
            d[f"csr_file_{i}"] = np.fromfile(path, np.uint8)
    np.savez_compressed(OUT, **d)
    print(OUT, os.path.getsize(OUT), "bytes,", len(d), "arrays")


if __name__ == "__main__":
    main()
