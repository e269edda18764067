"""GPU suite (-m gpu): betweenness centrality through ess.bc / ess_bc / bc::run.

Values are compared with the float64 restatement tests/bc_ref.py at rtol 1e-5 (the library sums in double and rounds
once to float32): exact all-sources BC on the golden graphs, a directed RMAT with a caller CSC and multigraphs with
parallel edges and self-loops; a graph whose in- and out-hubs (>= 4096 edges) and warp-sized rows reach every gather
mode. The result is a pure function of (graph, sources, scale), so repeated runs, 32- and 64-bit offsets, host-built
and misaligned graphs must agree byte for byte, and sources=[s, s] must be exactly twice sources=[s]. On Kronecker
scale-20 the sum of the dependencies is checked against the BFS depths, a certificate that needs no CPU reference."""
import importlib.util
import math
import os
from ctypes import byref, c_int32, c_void_p

import numpy as np
import pytest
import torch

import bc_ref as ref
import essentials_b200 as ess
import oracle
from essentials_b200 import graphgen as gg

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INT_MAX = 2**31 - 1


def _load_cost_script():
    spec = importlib.util.spec_from_file_location("bc_cost", os.path.join(ROOT, "scripts", "bc_cost.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


certificate = _load_cost_script().certificate  # the check the cost measurement applies to every timed source


@pytest.fixture(scope="module")
def ctx():
    assert torch.cuda.is_available(), "GPU suite needs a CUDA device"
    return ess.Context(0)


def _dev(a, dtype):
    return torch.from_numpy(np.ascontiguousarray(a).astype(dtype)).cuda()


def _csr(off, col, name, symmetric, wide=False):
    return gg.CSR(len(off) - 1, len(col), _dev(off, np.int64 if wide else np.int32), _dev(col, np.int32), None, name,
                  symmetric)


def _directed(n, src, dst, name, wide=False):
    """CSR of src -> dst and its transpose as the caller CSC, built on the host."""
    off, col = ref.from_edges(n, src, dst)
    toff, tcol = ref.from_edges(n, dst, src)
    csr, csc = _csr(off, col, name, False, wide), _csr(toff, tcol, name + "-T", False, wide)
    return off, col, ess.Graph(csr, csc=csc)


def _close(got, want, what):
    got = got.cpu().numpy().astype(np.float64)
    assert np.isfinite(got).all(), what
    assert np.allclose(got, want, rtol=1e-5, atol=0), (what, np.abs(got - want).max())


# ------------------------------------------------------------------------------------------------ values
def test_exact_bc_on_the_golden_graphs(ctx, golden):
    for name, gd in golden.items():
        off, col = gd["offsets"], gd["indices"]
        g = ess.Graph(_csr(off, col, name, True))
        got, info = ess.bc(ctx, g)
        assert info["sources"] == g.n
        _close(got, ref.brandes(off, col), name)
        g.close()


def test_exact_bc_on_a_directed_rmat_with_a_caller_csc(ctx):
    csr = gg.rmat_csr(9, symmetric=False, device="cuda")
    g = ess.Graph(csr, csc=ess.transpose(csr))
    off, col, _ = csr.host()
    got, _ = ess.bc(ctx, g)
    _close(got, ref.brandes(off, col), "directed rmat-9")


@pytest.mark.parametrize("symmetric", [False, True])
def test_exact_bc_on_multigraphs_with_parallel_edges_and_self_loops(ctx, symmetric):
    rng = np.random.default_rng(31 + symmetric)
    for trial in range(12):
        n, src, dst = ref.random_multigraph(rng, symmetric)
        if symmetric:
            off, col = ref.from_edges(n, src, dst)
            g = ess.Graph(_csr(off, col, "multigraph", True))
        else:
            off, col, g = _directed(n, src, dst, "multigraph")
        got, _ = ess.bc(ctx, g)
        _close(got, ref.brandes(off, col), (trial, symmetric))
        sub = [int(s) for s in rng.integers(0, n, 4)]
        _close(ess.bc(ctx, g, sub, scale=0.5)[0], ref.brandes(off, col, sub, 0.5), (trial, sub))
        g.close()


def test_every_gather_mode(ctx):
    """A directed graph with an out-hub (5000 out-edges), an in-hub (6000 in-edges), rows of 8..200 edges both ways
    and a sparse background: thread, warp and CTA rows in the forward and the backward pass."""
    rng = np.random.default_rng(7)
    n = 30000
    src = [rng.integers(0, n, 60000)]
    dst = [rng.integers(0, n, 60000)]
    src.append(np.full(5000, 3)), dst.append(rng.integers(0, n, 5000))  # out-hub 3
    src.append(rng.integers(0, n, 6000)), dst.append(np.full(6000, 11))  # in-hub 11
    mid = rng.integers(0, n, 300)
    for v in mid:
        k = int(rng.integers(8, 200))
        src += [np.full(k, v), rng.integers(0, n, k)]
        dst += [rng.integers(0, n, k), np.full(k, v)]
    src.append(np.array([11, 11])), dst.append(np.array([3, 11]))  # in-hub -> out-hub, a self-loop on the in-hub
    src, dst = np.concatenate(src), np.concatenate(dst)
    off, col, g = _directed(n, src, dst, "hubs")
    indeg, outdeg = np.bincount(dst, minlength=n), np.diff(off)
    sources = [3, 11, int(mid[0]), 0, int(np.argmax(outdeg == 1))]
    depth = ref.depths(n, *ref.edge_list(off, col), 0)
    assert depth[3] > 0 and depth[11] > 0, "both hubs are reached from source 0"
    reached = depth >= 0
    for deg in (indeg, outdeg):  # every bin is populated among the reached vertices
        assert (reached & (deg < 8)).any() and (reached & (deg >= 8) & (deg < 4096)).any() and (
            reached & (deg >= 4096)).any()
    got, info = ess.bc(ctx, g, sources)
    _close(got, ref.brandes(off, col, sources), "hubs")
    assert info["sources"] == len(sources) and info["reached"] > 0 and info["edges_gathered"] > 0


# ------------------------------------------------------------------------------------------------ byte identity
def _misaligned(t):
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    view = buf[1:]
    view.copy_(t)
    assert view.data_ptr() % 16 == t.element_size()
    return view


def test_byte_identical_across_runs_and_graph_builds(ctx):
    csr = gg.rmat_csr(13, device="cuda")
    sources = gg.pick_sources(csr, 4)
    g = ess.Graph(csr)
    base, _ = ess.bc(ctx, g, sources)
    assert torch.equal(ess.bc(ctx, g, sources)[0], base), "two runs"
    wide = gg.CSR(csr.n, csr.m, csr.offsets.long(), csr.indices, None, csr.name, True)
    gw = ess.Graph(wide)
    assert torch.equal(ess.bc(ctx, gw, sources)[0], base), "int64 offsets"
    gh = ess.Graph.from_host(ctx, csr.to("cpu"))
    assert torch.equal(ess.bc(ctx, gh, sources)[0], base), "from_host"
    mis = gg.CSR(csr.n, csr.m, _misaligned(csr.offsets), _misaligned(csr.indices), None, csr.name, True)
    gm = ess.Graph(mis)
    assert torch.equal(ess.bc(ctx, gm, sources)[0], base), "misaligned arrays"
    s = sources[0]
    one, _ = ess.bc(ctx, g, s)
    two, info = ess.bc(ctx, g, [s, s])
    assert info["sources"] == 2
    assert torch.equal(two, 2 * one), "a source listed twice counts twice"
    assert torch.equal(ess.bc(ctx, g, torch.tensor([s, s], dtype=torch.int64))[0], two), "CPU tensor of sources"
    for h in (gw, gh, gm, g):
        h.close()


def test_scale_is_honoured(ctx):
    csr = gg.rmat_csr(11, device="cuda")
    g = ess.Graph(csr)
    sources = gg.pick_sources(csr, 3)
    raw, _ = ess.bc(ctx, g, sources)
    assert torch.equal(ess.bc(ctx, g, sources, scale=0.25)[0], raw * 0.25)
    norm = 1.0 / ((g.n - 1) * (g.n - 2))
    off, col, _ = csr.host()
    _close(ess.bc(ctx, g, sources, scale=norm)[0], ref.brandes(off, col, sources, norm), "normalised")
    assert torch.count_nonzero(ess.bc(ctx, g, sources, scale=0.0)[0]) == 0


# ------------------------------------------------------------------------------------------------ buffers, errors
def test_caller_out_buffer(ctx):
    csr = gg.rmat_csr(10, device="cuda")
    g = ess.Graph(csr)
    want, _ = ess.bc(ctx, g, [1, 2])
    out = torch.full((g.n + 5,), float("nan"), device="cuda")
    got, _ = ess.bc(ctx, g, [1, 2], out=out)
    assert got.data_ptr() == out.data_ptr() and torch.equal(out[:g.n], want), "garbage is overwritten"
    assert torch.isnan(out[g.n:]).all(), "nothing past n is written"
    for bad in (torch.empty(g.n - 1, device="cuda"), torch.empty(g.n, dtype=torch.float64, device="cuda"),
                torch.empty(g.n), torch.empty(2 * g.n, device="cuda")[::2]):
        with pytest.raises(ess.EssentialsError, match="float32 CUDA tensor"):
            ess.bc(ctx, g, [1], out=bad)


def test_errors(ctx):
    csr = gg.rmat_csr(8, symmetric=False, device="cuda")
    g = ess.Graph(csr)
    assert not g.has_csc
    with pytest.raises(ess.EssentialsError, match="CSR and CSC sparse-matrix representations required"):
        ess.bc(ctx, g, [0])
    gs = ess.Graph(gg.rmat_csr(8, device="cuda"))
    with pytest.raises(ess.EssentialsError, match="out of range"):
        ess.bc(ctx, gs, [gs.n])
    # the C ABI refuses the same inputs on its own, before any launch
    out = torch.full((gs.n,), 7.0, device="cuda")
    L = ess.lib()

    def call(sources, count, scale=1.0, d_bc=c_void_p(out.data_ptr()), graph=gs.handle):
        arr = (c_int32 * max(len(sources), 1))(*sources)
        info = ess.RunInfo()
        return L.ess_bc(ctx.handle, graph, arr if sources else None, count, scale, d_bc, byref(info))

    assert call([gs.n], 1) != 0 and b"out of range" in L.ess_last_error()
    assert call([-1], 1) != 0 and b"out of range" in L.ess_last_error()
    assert call([], -1) != 0 and b"negative" in L.ess_last_error()
    assert call([0], 0) != 0 and b"NULL" in L.ess_last_error()
    assert call([0], 1, scale=math.inf) != 0 and b"finite" in L.ess_last_error()
    assert call([0], 1, scale=math.nan) != 0 and b"finite" in L.ess_last_error()
    assert call([0], 1, d_bc=None) != 0 and b"null" in L.ess_last_error()
    assert call([0], 1, graph=g.handle) != 0 and b"CSC" in L.ess_last_error()
    torch.cuda.synchronize()
    assert bool((out == 7.0).all()), "a refused call writes nothing"


# ------------------------------------------------------------------------------------------------ the reference
@pytest.mark.skipif(not oracle.have_ref_on_ours(), reason="oracle/_ref/libref_algos_on_ours.so not built")
def test_single_source_matches_the_reference_bc(ctx):
    """The reference's bc.hxx on our operators returns scale 0.5 on v != s; its own value at s is not compared."""
    csr = gg.rmat_csr(9, weights="ones", device="cuda")
    g = ess.Graph(csr)
    for s in gg.pick_sources(csr, 2):
        want, _ = oracle.ref_on_ours_extra("bc", csr, s)
        got, _ = ess.bc(ctx, g, s, scale=0.5)
        assert float(got[s]) == 0.0
        w, o = want.cpu().numpy().astype(np.float64), got.cpu().numpy().astype(np.float64)
        w[s] = o[s] = 0.0
        assert np.allclose(o, w, rtol=1e-4, atol=1e-4), s


# ------------------------------------------------------------------------------------------------ certificate
def test_kronecker_scale20_certificate(ctx):
    csr = gg.rmat_csr(20, device="cuda")
    g = ess.Graph(csr)
    degree = csr.degrees().to("cuda")  # a simple graph: the degree is the number of distinct neighbours
    for s in gg.pick_sources(csr, 4):
        got, info = ess.bc(ctx, g, [s])
        depth, _ = ess.bfs(ctx, g, s, lb="merge_path", direction="optimized")
        c = certificate(got, depth, s, degree)
        assert c["rel_err"] <= 1e-6 and c["negative"] == 0 and c["leaf_nonzero"] == 0, (s, c)
        assert info["reached"] == int((depth != INT_MAX).sum())
