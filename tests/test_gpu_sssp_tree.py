"""GPU suite (-m gpu): the SSSP tree of ess.sssp_tree / ess_sssp_tree / sssp::build_tree.

The tree is a pure function of the graph, the distances and the source (include/essentials_b200.h states the rules), so
every test demands exact equality: with the CPU restatement tests/sssp_tree_ref.cpp on the same distances, and between
the trees built from the distances of every SSSP engine (ess.sssp with every balancer, ess.sssp_near_far,
ess.sssp_delta). Inputs: the golden graphs, arbitrary directed multigraphs given as CSR only, a 5000-edge zero-weight
chain, extreme weight ranges, int64 offsets, graphs built from host arrays, misaligned graph arrays, the scalar advance
kernels, and caller buffers that hold garbage, start 4 bytes past a 16-byte boundary or are reused. Distances that are
not the SSSP fixed point must be refused with a message naming the violation, and host-side argument errors must be
refused before any kernel is launched."""
import dataclasses
import importlib.util
import os
from ctypes import byref, c_void_p

import numpy as np
import pytest
import torch

import essentials_b200 as ess
import oracle
import sssp_tree_ref as ref
from essentials_b200 import graphgen as gg
from test_sssp_tree_oracle import arbitrary_multigraph, forged_distances, forged_graph, from_edges, numpy_tree

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LBS = list(ess.IMPLEMENTED_LOAD_BALANCERS)
KNOB_DEFAULTS = {"advance_engine": 1}


def _load_cost_script():
    spec = importlib.util.spec_from_file_location("sssp_tree_cost", os.path.join(ROOT, "scripts", "sssp_tree_cost.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


sssp_tree_violations = _load_cost_script().sssp_tree_violations  # the checker the cost measurement uses


@pytest.fixture(scope="module")
def ctx():
    assert torch.cuda.is_available(), "GPU suite needs a CUDA device"
    return ess.Context(0)


class knob:
    """ess.tune(name, value) for the duration of a with-block; the default is restored however the block ends."""

    def __init__(self, name, value):
        self.name, self.value = name, value

    def __enter__(self):
        ess.tune(self.name, self.value)

    def __exit__(self, *exc):
        ess.tune(self.name, KNOB_DEFAULTS[self.name])


def _misaligned(t):
    """Copy of `t` in a view one element into a fresh buffer: 4 bytes past a 16-byte boundary for 4-byte types."""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    view = buf[1:]
    view.copy_(t)
    assert view.data_ptr() % 16 == 4
    return view


def _csr(off, col, val, name, symmetric=False):
    return gg.CSR(off.size - 1, col.size, torch.from_numpy(off.astype(np.int32)).cuda(),
                  torch.from_numpy(col.astype(np.int32)).cuda(),
                  None if val is None else torch.from_numpy(val.astype(np.float32)).cuda(), name, symmetric)


def expected(off, col, w, s, d):
    pred, status = ref.sssp_tree(off, col, w, s, d)
    assert status == ref.OK, ref.STATUS[status]
    return pred


def tree_equals(ctx, g, s, dist, want, **kw):
    before = dist.clone()
    pred, info = ess.sssp_tree(ctx, g, s, dist, **kw)
    assert torch.equal(dist, before), "sssp_tree must not write dist"
    assert np.array_equal(pred[:want.size].cpu().numpy(), want), s
    return pred, info


# ------------------------------------------------------------------------------------------------ golden graphs
def test_golden_trees_are_byte_identical_across_engines(ctx, golden):
    """chesapeake, rmat_s10, grid_24x17 from every golden source: the trees built from the distances of every engine
    and balancer equal the tree of the golden distances."""
    for name, gd in golden.items():
        csr = _csr(gd["offsets"], gd["indices"], gd["values"], name, True)
        off, col, val = csr.host()
        g = ess.Graph(csr)
        for s in gd["sources"]:
            s = int(s)
            want_d = gd[f"sssp_{s}"]
            want = expected(off, col, val, s, want_d)
            runs = {f"sssp {lb}": ess.sssp(ctx, g, s, lb=lb)[0] for lb in LBS}
            runs["near_far"] = ess.sssp_near_far(ctx, g, s)[0]
            runs["near_far delta 2"] = ess.sssp_near_far(ctx, g, s, delta=2.0)[0]
            runs["delta"] = ess.sssp_delta(ctx, g, s)[0]
            for what, dist in runs.items():
                assert np.array_equal(dist.cpu().numpy(), want_d), (name, s, what)
                tree_equals(ctx, g, s, dist, want)
        g.close()


# ------------------------------------------------------------------------------------------------ flat edges
def test_arbitrary_directed_multigraphs_without_csc(ctx):
    """Self loops, parallel edges, isolated vertices, zero weights and weights absorbed next to 1e8, CSR only. The flat
    rounds must equal the deepest flat hop count of the numpy restatement."""
    rng = np.random.default_rng(51)
    deepest = 0
    for trial in range(60):
        n, off, col, w = arbitrary_multigraph(rng)
        g = ess.Graph(_csr(off, col, w, "arbitrary"))
        assert not g.has_csc
        for s in {0, int(rng.integers(0, n)), n - 1}:
            want_d = oracle.sssp(off, col, w, s)
            want, rounds = numpy_tree(off, col, w, s, want_d)
            assert np.array_equal(want, expected(off, col, w, s, want_d))
            for dist in (ess.sssp(ctx, g, s, lb="merge_path")[0], ess.sssp_delta(ctx, g, s)[0],
                         ess.sssp_near_far(ctx, g, s)[0]):
                assert np.array_equal(dist.cpu().numpy(), want_d), (trial, s)
                _, info = tree_equals(ctx, g, s, dist, want)
                assert info["flat_rounds"] == rounds, (trial, s, info["flat_rounds"], rounds)
            deepest = max(deepest, rounds)
        g.close()
    assert deepest > 0


def test_flat_rounds_follow_a_long_zero_weight_chain(ctx):
    """0 -1-> 1, then 5000 zero-weight edges 1 -> 2 -> ... -> 5001 and a zero-weight cycle 5001 -> 5002 -> 5003 ->
    5001, with weighted shortcuts that lose: one flat round per hop."""
    chain = 5000
    src = [0] + list(range(1, chain + 1)) + [chain + 1, chain + 2, chain + 3, 0, 0]
    dst = [1] + list(range(2, chain + 2)) + [chain + 2, chain + 3, chain + 1, chain + 1, 2500]
    w = [1.0] + [0.0] * chain + [0.0, 0.0, 0.0, 2.0, 1.5]
    n = chain + 5  # the last vertex is isolated
    off, col, w = from_edges(n, np.array(src), np.array(dst), np.array(w))
    g = ess.Graph(_csr(off, col, w, "chain"))
    want_d = oracle.sssp(off, col, w, 0)
    want, rounds = numpy_tree(off, col, w, 0, want_d)
    assert rounds >= chain
    for dist in (ess.sssp(ctx, g, 0, lb="merge_path")[0], ess.sssp_delta(ctx, g, 0)[0]):
        assert np.array_equal(dist.cpu().numpy(), want_d)
        _, info = tree_equals(ctx, g, 0, dist, want)
        assert info["flat_rounds"] == rounds and info["flat_rounds"] >= chain, info
        assert info["flat_vertices"] == chain + 2, info


def test_extreme_weight_ranges(ctx):
    """The {1e-3, 1e6} grid: distances of millions absorb the 1e-3 steps into flat edges, so the flat rounds run
    (14 and 4 of them from these sources)."""
    grid = gg.grid_csr(40, 30, device="cuda")
    rows = torch.repeat_interleave(torch.arange(grid.n, device="cuda"), grid.degrees().long())
    lo, hi = torch.minimum(rows, grid.indices.long()), torch.maximum(rows, grid.indices.long())
    w = torch.where(((lo * 31 + hi) % 5) == 0, 1e6, 1e-3).to(torch.float32)
    g2 = dataclasses.replace(grid, values=w)
    off, col, val = g2.host()
    g = ess.Graph(g2)
    for s in (0, grid.n // 2 + 7):
        want_d = oracle.sssp(off, col, val, s)
        want, rounds = numpy_tree(off, col, val, s, want_d)
        assert rounds > 0
        assert np.array_equal(want, expected(off, col, val, s, want_d))
        for dist in (ess.sssp_near_far(ctx, g, s, delta=1e-3)[0], ess.sssp_delta(ctx, g, s, delta=1e-3)[0],
                     ess.sssp(ctx, g, s, lb="block_mapped")[0]):
            assert np.array_equal(dist.cpu().numpy(), want_d)
            _, info = tree_equals(ctx, g, s, dist, want)
            assert info["flat_rounds"] == rounds, (s, info)


# ------------------------------------------------------------------------------------------------ graph inputs
@pytest.fixture(scope="module")
def s16():
    """Directed weighted RMAT scale 16 with int64 offsets; a third of the edges weigh 0, so flat rounds run."""
    csr = gg.rmat_csr(16, symmetric=False, weights="hash", device="cuda", offset_bits=64)
    csr = dataclasses.replace(csr, values=torch.where(csr.indices % 3 == 0, 0.0, csr.values))
    assert csr.offsets.dtype == torch.int64
    return csr, csr.host()


def _sources(csr):
    return [0] + gg.pick_sources(csr, 2)


def _check_graph(ctx, g, csr, host, engines=("delta", "merge_path")):
    off, col, val = host
    flat = 0
    for s in _sources(csr):
        want_d = oracle.sssp(off, col, val, s)
        want = expected(off, col, val, s, want_d)
        for engine in engines:
            dist = ess.sssp_delta(ctx, g, s)[0] if engine == "delta" else ess.sssp(ctx, g, s, lb=engine)[0]
            assert np.array_equal(dist.cpu().numpy(), want_d), (s, engine)
            _, info = tree_equals(ctx, g, s, dist, want)
            flat = max(flat, info["flat_rounds"])
    return flat


def test_rmat16_int64_offsets(ctx, s16):
    csr, host = s16
    assert _check_graph(ctx, ess.Graph(csr), csr, host, ("delta",) + tuple(LBS)) > 0


def test_graphs_from_host_arrays(ctx, s16):
    csr, host = s16
    narrow = dataclasses.replace(csr, offsets=csr.offsets.int())
    for what, c in (("int32", narrow), ("int64", csr)):
        g = ess.Graph.from_host(ctx, c.pinned(), symmetric=False)
        assert g.offset_bits == (32 if what == "int32" else 64)
        _check_graph(ctx, g, csr, host)
        g.close()


def test_misaligned_graph_arrays(ctx, s16):
    """Column indices and values 4 bytes past a 16-byte boundary: the sweep takes the scalar advance kernels."""
    csr, host = s16
    odd = dataclasses.replace(csr, indices=_misaligned(csr.indices), values=_misaligned(csr.values))
    _check_graph(ctx, ess.Graph(odd), csr, host)


def test_scalar_advance_kernels(ctx, s16):
    csr, host = s16
    g = ess.Graph(csr)
    with knob("advance_engine", 0):
        _check_graph(ctx, g, csr, host)


# ------------------------------------------------------------------------------------------------ caller buffers
def test_caller_buffers(ctx, s16):
    """pred_out full of garbage (the source's id, ids past n, negative ids), misaligned views of both arrays, and one
    buffer reused across sources: the result never depends on what the buffer held, and dist is never written."""
    csr, (off, col, val) = s16
    g = ess.Graph(csr)
    gen = torch.Generator(device="cuda").manual_seed(7)
    shared = torch.empty(csr.n, dtype=torch.int32, device="cuda")
    for s in _sources(csr):
        want_d = oracle.sssp(off, col, val, s)
        want = expected(off, col, val, s, want_d)
        dist, _ = ess.sssp_delta(ctx, g, s)
        garbage = torch.randint(-2**31, 2**31 - 1, (csr.n,), dtype=torch.int32, device="cuda", generator=gen)
        garbage[::5] = s
        garbage[1::5] = csr.n + 3
        pred, _ = tree_equals(ctx, g, s, dist, want, pred_out=garbage)
        assert pred.data_ptr() == garbage.data_ptr()
        odd_pred = _misaligned(torch.full((csr.n,), s, dtype=torch.int32, device="cuda"))
        pred, _ = tree_equals(ctx, g, s, _misaligned(dist), want, pred_out=odd_pred)
        assert pred.data_ptr() == odd_pred.data_ptr()
        pred, _ = tree_equals(ctx, g, s, dist, want, pred_out=shared)
        assert pred.data_ptr() == shared.data_ptr()
    longer = torch.full((csr.n + 9,), 77, dtype=torch.int32, device="cuda")
    s = _sources(csr)[-1]
    tree_equals(ctx, g, s, ess.sssp_delta(ctx, g, s)[0], expected(off, col, val, s, oracle.sssp(off, col, val, s)),
                pred_out=longer)
    assert (longer[csr.n:] == 77).all(), "entries past n are not the tree's"


# ------------------------------------------------------------------------------------------------ errors
def test_host_side_errors_are_raised_before_any_launch(ctx, s16):
    csr, _ = s16
    n = csr.n
    g = ess.Graph(csr)
    dist, _ = ess.sssp_delta(ctx, g, 0)
    buf = torch.zeros(2 * n, dtype=torch.int32, device="cuda")
    bad = {
        "source -1": dict(source=-1),
        "source n": dict(source=n),
        "pred_out overlaps dist": dict(dist=buf[n // 2: n // 2 + n].view(torch.float32), pred_out=buf[:n]),
        "pred_out is dist": dict(pred_out=dist.view(torch.int32)),
        "float64 dist": dict(dist=dist.double()),
        "int32 dist": dict(dist=dist.view(torch.int32)),
        "int64 pred_out": dict(pred_out=torch.empty(n, dtype=torch.int64, device="cuda")),
        "float32 pred_out": dict(pred_out=torch.empty(n, dtype=torch.float32, device="cuda")),
        "short dist": dict(dist=dist[:n - 1]),
        "short pred_out": dict(pred_out=torch.empty(n - 1, dtype=torch.int32, device="cuda")),
        "host dist": dict(dist=dist.cpu()),
        "host pred_out": dict(pred_out=torch.empty(n, dtype=torch.int32)),
        "strided dist": dict(dist=torch.empty(2 * n, dtype=torch.float32, device="cuda")[::2]),
        "strided pred_out": dict(pred_out=torch.empty(2 * n, dtype=torch.int32, device="cuda")[::2]),
        "dist is a list": dict(dist=[0.0] * n),
    }
    for what, kw in bad.items():
        s = kw.pop("source", 0)
        d = kw.pop("dist", dist)
        launches = ctx.launches()
        with pytest.raises(ess.EssentialsError):
            ess.sssp_tree(ctx, g, s, d, **kw)
        assert ctx.launches() == launches, what
    # the C ABI's own checks (the binding stops these before the call)
    info = ess.RunInfo()
    L = ess.lib()
    pd, pp = c_void_p(dist.data_ptr()), c_void_p(buf.data_ptr())
    for args, message in (((0, None, pp), b"null"), ((0, pd, None), b"null"), ((0, pd, pd), b"overlap"),
                          ((0, pd, c_void_p(dist.data_ptr() + 4 * (n - 1))), b"overlap"),
                          ((0, c_void_p(buf.data_ptr() + 4 * (n - 1)), pp), b"overlap"),
                          ((n, pd, pp), b"out of range"), ((-1, pd, pp), b"out of range")):
        launches = ctx.launches()
        assert L.ess_sssp_tree(ctx.handle, g.handle, *args, byref(info)) != 0
        assert message in L.ess_last_error(), (args, L.ess_last_error())
        assert ctx.launches() == launches
    assert L.ess_sssp_tree(None, g.handle, 0, pd, pp, byref(info)) != 0
    assert L.ess_sssp_tree(ctx.handle, None, 0, pd, pp, byref(info)) != 0


MESSAGES = {ref.INVALID_ENTRY: "NaN, negative or infinite", ref.SOURCE_NOT_ZERO: "source's distance is not 0",
            ref.RELAXABLE_EDGE: "relaxable edges", ref.ORPHAN: "reached vertices have no tight path from the source"}


def test_forged_distances_are_refused_on_the_device(ctx):
    """Each forged array of the CPU test raises with a message naming its violation; the context stays usable."""
    off, col, w = forged_graph()
    g = ess.Graph(_csr(off, col, w, "forged"))
    good = oracle.sssp(off, col, w, 0)
    for name, (x, status) in forged_distances().items():
        with pytest.raises(ess.EssentialsError, match=MESSAGES[status]):
            ess.sssp_tree(ctx, g, 0, torch.from_numpy(x).cuda())
        tree_equals(ctx, g, 0, torch.from_numpy(good).cuda(), expected(off, col, w, 0, good))
    counts = {"lowered": "1 reached vertices", "unreachable zero-weight cycle": "2 reached vertices",
              "raised": "1 relaxable edges", "reached vertex marked FLT_MAX": "3 relaxable edges",
              "NaN": "1 entries are NaN"}
    cases = forged_distances()
    for name, text in counts.items():
        with pytest.raises(ess.EssentialsError, match=text):
            ess.sssp_tree(ctx, g, 0, torch.from_numpy(cases[name][0]).cuda())


# ------------------------------------------------------------------------------------------------ Kronecker scale 20
def test_kronecker20_tree_on_the_device(ctx):
    """Weighted Kronecker scale 20: the checker the cost measurement uses reports nothing, and the tree equals the CPU
    restatement."""
    csr = gg.rmat_csr(20, weights="hash", device="cuda")
    g = ess.Graph(csr)
    off, col, val = csr.host()
    for s in gg.pick_sources(csr, 2):
        dist, _ = ess.sssp_delta(ctx, g, s)
        pred, info = ess.sssp_tree(ctx, g, s, dist)
        v = sssp_tree_violations(csr.offsets, csr.indices, csr.values, s, dist, pred, chunk=1 << 22)
        assert not any(v.values()), (s, v)
        assert info["flat_rounds"] == 0
        assert np.array_equal(pred.cpu().numpy(), expected(off, col, val, s, dist.cpu().numpy())), s
    g.close()
