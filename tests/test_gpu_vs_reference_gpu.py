"""GPU suite: our CUDA path vs the REFERENCE's own GPU implementation (oracle/_ref/libref_gpu.so: the reference's
algorithm headers + block_mapped advance + Thrust filters compiled for sm_100 from the reference's sources) on the same
inputs; where that build is absent, BFS, SSSP and k-core are compared with its stored outputs
(tests/golden/reference_outputs.npz). BFS depths, SSSP distances (bit-exact), k-core numbers identical; PageRank / PPR within tolerance;
colouring is checked for validity only, like the reference driver (its device random stream uses fast-math)."""
import os

import numpy as np
import pytest
import torch

import essentials_b200 as ess
import oracle
from essentials_b200 import graphgen as gg

pytestmark = pytest.mark.gpu
needs_ref_gpu = pytest.mark.skipif(not oracle.have_ref_gpu(), reason="oracle/_ref/libref_gpu.so not built")
# BFS depths, SSSP distances and core numbers the reference returns on these inputs (one right answer each;
# tests/golden/make_reference_vectors.py), compared with where the reference's GPU build is absent
STORED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.npz")


def _reference(alg, csr, key, *params):
    """The reference GPU implementation's output: run it when built, else its stored output for this input."""
    if oracle.have_ref_gpu():
        return oracle.ref_gpu_run(alg, csr, *params)[0]
    return torch.from_numpy(np.load(STORED)[key]).to(csr.indices.device)


@pytest.fixture(scope="module")
def ctx():
    return ess.Context(0)


@pytest.fixture(scope="module")
def kron():
    csr = gg.rmat_csr(15, weights="hash", device="cuda")
    return csr, ess.Graph(csr)


def test_bfs_equals_reference_gpu(ctx, kron):
    csr, g = kron
    sources = [0] + gg.pick_sources(csr, 2)
    assert oracle.have_ref_gpu() or sources == np.load(STORED)["kron15_sources"].tolist()
    for s in sources:
        want = _reference("bfs", csr, f"kron15_bfs_{s}", s)
        for lb, direction in (("block_mapped", "forward"), ("merge_path", "optimized"), ("bucketing", "forward")):
            got, _ = ess.bfs(ctx, g, s, lb=lb, direction=direction)
            assert torch.equal(got, want), (s, lb, direction)


def test_sssp_equals_reference_gpu(ctx, kron):
    csr, g = kron
    s = gg.pick_sources(csr, 1)[0]
    want = _reference("sssp", csr, f"kron15_sssp_{s}", s)
    for lb in ("block_mapped", "merge_path"):
        got, _ = ess.sssp(ctx, g, s, lb=lb)
        assert torch.equal(got, want), lb


def test_kcore_equals_reference_gpu(ctx):
    csr = gg.rmat_csr(11, device="cuda")
    want = _reference("kcore", csr, "kron11_kcore")
    got, _ = ess.kcore(ctx, ess.Graph(csr), lb="merge_path")
    assert torch.equal(got, want)


@needs_ref_gpu
def test_pagerank_and_ppr_close_to_reference_gpu(ctx):
    csr = gg.rmat_csr(12, symmetric=False, weights="ones", device="cuda")
    want, _ = oracle.ref_gpu_run("pr", csr, 0.85, 1e-6)
    g = ess.Graph(csr, csc=ess.transpose(csr))
    for pull in (False, True):
        got, _ = ess.pagerank(ctx, g, lb="merge_path", pull=pull)
        rel = ((got.double() - want.double()).abs().sum() / want.double().sum()).item()
        assert rel < 2e-6, (pull, rel)  # both sides sum floats in a different, unordered way
    sym = gg.rmat_csr(11, device="cuda")
    want, _ = oracle.ref_gpu_run("ppr", sym, 3, 0.15, 1e-6)
    got, _ = ess.ppr(ctx, ess.Graph(sym), 3)
    assert float((got - want).abs().max()) <= 1e-6


@needs_ref_gpu
def test_reference_gpu_colouring_is_valid_and_ours_too(ctx, kron):
    csr, g = kron
    off, col, _ = csr.host()
    ref_colors, _ = oracle.ref_gpu_run("color", csr)
    ours, _ = ess.color(ctx, g)
    assert oracle.color_errors(off, col, ref_colors.cpu().numpy()) == 0
    assert oracle.color_errors(off, col, ours.cpu().numpy()) == 0


# ---- the reference's UNMODIFIED algorithm headers compiled against our operator headers ----------------------
needs_compat = pytest.mark.skipif(not oracle.have_ref_on_ours(), reason="oracle/_ref/libref_algos_on_ours.so not built")


@needs_compat
def test_reference_algorithm_headers_run_on_our_operators(ctx, kron):
    """Drop-in proof: reference bfs/sssp/kcore/pr/ppr/color sources + our include tree == all-reference build."""
    csr, g = kron
    off, col, val = csr.host()
    s = gg.pick_sources(csr, 1)[0]
    ref_bfs, _ = oracle.ref_gpu_run("bfs", csr, s)
    got, _ = oracle.ref_gpu_run("bfs", csr, s, on_ours=True)
    assert torch.equal(got, ref_bfs)
    assert np.array_equal(got.cpu().numpy(), oracle.bfs(off, col, s))
    ref_sssp, _ = oracle.ref_gpu_run("sssp", csr, s)
    got, _ = oracle.ref_gpu_run("sssp", csr, s, on_ours=True)
    assert torch.equal(got, ref_sssp)
    small = gg.rmat_csr(11, device="cuda")
    assert torch.equal(oracle.ref_gpu_run("kcore", small, on_ours=True)[0], oracle.ref_gpu_run("kcore", small)[0])
    got, _ = oracle.ref_gpu_run("ppr", small, 3, 0.15, 1e-6, on_ours=True)
    want, _ = oracle.ref_gpu_run("ppr", small, 3, 0.15, 1e-6)
    assert float((got - want).abs().max()) <= 1e-6
    directed = gg.rmat_csr(12, symmetric=False, weights="ones", device="cuda")
    got, _ = oracle.ref_gpu_run("pr", directed, 0.85, 1e-6, on_ours=True)
    want, _ = oracle.ref_gpu_run("pr", directed, 0.85, 1e-6)
    assert ((got.double() - want.double()).abs().sum() / want.double().sum()).item() < 2e-6
    o, c, _ = small.host()
    colors, _ = oracle.ref_gpu_run("color", small, on_ours=True)
    assert oracle.color_errors(o, c, colors.cpu().numpy()) == 0
    assert np.array_equal(colors.cpu().numpy(), oracle.color_jacobi(o, c)[0]), "our random stream + deterministic filter"


def _brandes_single_source(off, col, s):
    """Dependency scores of one source (Brandes), the quantity gunrock::bc::run(G, source, bc) accumulates."""
    n = off.size - 1
    depth = oracle.bfs(off, col, s)
    order = np.argsort(depth, kind="stable")
    order = order[depth[order] != 2**31 - 1]
    sigma = np.zeros(n)
    sigma[s] = 1
    for v in order:
        for u in col[off[v]:off[v + 1]]:
            if depth[u] == depth[v] + 1:
                sigma[u] += sigma[v]
    delta = np.zeros(n)
    for v in order[::-1]:
        for u in col[off[v]:off[v + 1]]:
            if depth[u] == depth[v] + 1:
                delta[v] += sigma[v] / sigma[u] * (1 + delta[u])
    return delta


@needs_compat
def test_reference_bc_and_spmv_headers_on_our_operators(ctx):
    """§8f rows: bc drives the explicit-buffers merge_path advance with a per-depth frontier array
    (reference bc.hxx:98-190); spmv's pull form drives neighborreduce (spmv.hxx:107-127)."""
    csr = gg.rmat_csr(9, weights="ones", device="cuda")
    off, col, val = csr.host()
    s = gg.pick_sources(csr, 1)[0]
    got, _ = oracle.ref_on_ours_extra("bc", csr, s)
    want = _brandes_single_source(off, col, s)
    want[s] = 0.0
    g = got.cpu().numpy().astype(np.float64)
    g[s] = 0.0
    # the reference accumulates 0.5 * delta per back-propagated edge ("scaled output", bc.hxx:168)
    assert np.allclose(g, want / 2, rtol=1e-4, atol=1e-4), "bc dependency scores (Brandes / 2)"
    weighted = gg.rmat_csr(10, weights="hash", device="cuda")
    x = torch.rand(weighted.n, device="cuda")
    y, _ = oracle.ref_on_ours_extra("spmv", weighted, x)
    rows = torch.repeat_interleave(torch.arange(weighted.n, device="cuda"), weighted.degrees().long())
    want = torch.zeros(weighted.n, device="cuda", dtype=torch.float64).index_add_(
        0, rows, (weighted.values.double() * x[weighted.indices.long()].double()))
    assert torch.allclose(y.double(), want, rtol=1e-5, atol=1e-5)


@needs_compat
def test_reference_tc_header_on_our_operators_golden_counts(ctx):
    """§8f row 4: the reference's tc.hxx (advance<block_mapped, forward, graph -> none> + graph_t::get_intersection_count,
    tc.hxx:99-103) on our operators must reproduce the reference's own golden counts
    (unittests/algorithms/tc.cuh:24-54 and :57-93, the only hard known answers in the reference's test tree), and
    agree with a dense-matrix triangle count on a Kronecker graph."""
    import dataclasses
    cases = [([0, 3, 5, 8, 10], [1, 2, 3, 0, 2, 0, 1, 3, 0, 2], [2, 1, 2, 1], 6),
             ([0, 4, 7, 10, 12], [0, 1, 2, 3, 0, 1, 2, 0, 1, 3, 0, 2], [2, 1, 2, 1], 6)]  # second: self loops ignored
    for off, col, per_vertex, total in cases:
        csr = gg.CSR(len(off) - 1, len(col), torch.tensor(off, dtype=torch.int32, device="cuda"),
                     torch.tensor(col, dtype=torch.int32, device="cuda"),
                     torch.zeros(len(col), dtype=torch.float32, device="cuda"), "tc-golden", True)
        (counts, all_triangles), _ = oracle.ref_on_ours_extra("tc", csr)
        assert counts.cpu().tolist() == per_vertex and all_triangles == total
    kron = gg.rmat_csr(9, weights="ones", device="cuda")
    (counts, all_triangles), _ = oracle.ref_on_ours_extra("tc", kron)
    a = torch.zeros(kron.n, kron.n, dtype=torch.float64, device="cuda")
    rows = torch.repeat_interleave(torch.arange(kron.n, device="cuda"), kron.degrees().long())
    a[rows, kron.indices.long()] = 1.0
    want = torch.diagonal(a @ a @ a) / 2  # closed walks of length 3 through v, each triangle counted twice
    assert torch.equal(counts.double(), want) and all_triangles == int(want.sum().item())


_MST_SNIPPET = """
import sys, numpy as np, torch, scipy.sparse as sp
from scipy.sparse.csgraph import minimum_spanning_tree
sys.path.insert(0, {root!r})
import oracle
from essentials_b200 import graphgen as gg
grid = gg.grid_csr(24, 17, device="cuda")
off, col, val = grid.host()
assert np.unique(val).size == grid.m // 2, "distinct weights keep Boruvka free of ties"
got, ms = oracle.ref_on_ours_extra("mst", grid)
want = minimum_spanning_tree(sp.csr_matrix((val.astype(np.float64), col, off), shape=(grid.n, grid.n))).sum()
print("MST", float(got.item()), float(want))
_, hits_ms = oracle.ref_on_ours_extra("hits", grid, 20)
print("HITS", hits_ms)
"""


@needs_compat
def test_reference_hits_and_mst_headers_on_our_operators():
    """§8f row 4: mst.hxx (edge frontier, filter<remove> explicit form, parallel_for over elements and vertices,
    get_source_vertex) and hits.hxx (advance<block_mapped, graph -> vertices>) of the reference, unmodified, on our
    operators. MST weight against scipy's Kruskal. Runs in a child process with a timeout: the reference's pointer
    jumping spins on the device if a root cycle ever formed, and that must not be able to hang the suite."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-c", _MST_SNIPPET.format(root=root)], capture_output=True, text=True,
                         timeout=120)
    assert out.returncode == 0, out.stdout[-1500:] + out.stderr[-1500:]
    line = [l for l in out.stdout.splitlines() if l.startswith("MST")][0].split()
    got, want = float(line[1]), float(line[2])
    assert abs(got - want) <= 1e-4 * want, (got, want)
    assert any(l.startswith("HITS") for l in out.stdout.splitlines())
