"""GPU suite (-m gpu): the BFS tree of ess.bfs_tree / ess_bfs_tree / bfs::run_tree.

Contract, for a run from `source` with `depth` exactly as ess.bfs returns it: pred[source] == source; pred[v] == -1
exactly where depth[v] == INT32_MAX; every other pred[v] is in [0, n), is the tail of an edge pred[v] -> v of the CSR
and has depth[pred[v]] == depth[v] - 1. Which valid parent is chosen is not deterministic, so the tests check these
rules, never a particular tree, and they compare the depths bit for bit with ess.bfs, the golden vectors or the
oracle. Every balancer runs forward and direction-optimised, including the fallback kernels (pull_hints 0,
advance_engine 0, a misaligned graph), on caller buffers that hold garbage, start 4 bytes past a
16-byte boundary or are reused across sources."""
import importlib.util
import os

import numpy as np
import pytest
import torch

import essentials_b200 as ess
import oracle
from essentials_b200 import graphgen as gg

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LBS = list(ess.IMPLEMENTED_LOAD_BALANCERS)
INT32_MAX = np.iinfo(np.int32).max
KNOB_DEFAULTS = {"advance_engine": 1, "pull_hints": 1, "sssp_fused_unique": 1}


def _load_cost_script():
    spec = importlib.util.spec_from_file_location("bfs_tree_cost", os.path.join(ROOT, "scripts", "bfs_tree_cost.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


tree_violations = _load_cost_script().tree_violations  # the device checker the cost measurement uses


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


def _csr(off, col, val, name, symmetric, device="cuda"):
    return gg.CSR(off.size - 1, col.size, torch.from_numpy(off.astype(np.int32)).to(device),
                  torch.from_numpy(col.astype(np.int32)).to(device),
                  None if val is None else torch.from_numpy(val.astype(np.float32)).to(device), name, symmetric)


def _from_edges(n, src, dst, w=None):
    order = np.lexsort((dst, src))
    off = np.zeros(n + 1, np.int64)
    np.add.at(off, src + 1, 1)
    return np.cumsum(off), dst[order], None if w is None else w[order]


def _arbitrary_multigraph(rng):
    """Small directed multigraph with self loops, parallel edges, isolated vertices, zero and tied weights."""
    n = int(rng.integers(2, 70))
    m = int(rng.integers(1, 400))
    src, dst = rng.integers(0, n, m), rng.integers(0, n, m)
    w = rng.choice(np.array([0.0, 0.5, 1.0, 1.0, 2.25, 7.0, 63.984375], np.float32), m)
    off, col, val = _from_edges(n, src, dst, w)
    return _csr(off, col, val, "arbitrary", False)


def check_tree(off, col, source, depth, pred):
    """The three contract rules on host arrays (off: n + 1 row offsets of the CSR, col: its column indices)."""
    n = off.size - 1
    depth, pred = np.asarray(depth), np.asarray(pred)
    assert pred[source] == source, ("pred[source]", int(pred[source]), source)
    unreached = depth == INT32_MAX
    assert np.array_equal(pred == -1, unreached), ("-1 exactly where unreached",
                                                   np.flatnonzero((pred == -1) != unreached)[:8])
    rest = ~unreached
    rest[source] = False
    v = np.flatnonzero(rest)
    u = pred[v].astype(np.int64)
    assert ((u >= 0) & (u < n)).all(), ("parent out of range", v[(u < 0) | (u >= n)][:8])
    assert (depth[u] == depth[v] - 1).all(), ("parent depth", v[depth[u] != depth[v] - 1][:8])
    keys = np.repeat(np.arange(n, dtype=np.int64), np.diff(off)) * n + col.astype(np.int64)
    assert np.isin(u * n + v, keys).all(), ("parent edge missing", v[~np.isin(u * n + v, keys)][:8])


def _run_and_check(ctx, g, off, col, s, want, lb, direction, **kw):
    depth, pred, info = ess.bfs_tree(ctx, g, s, lb=lb, direction=direction, **kw)
    d = depth.cpu().numpy()
    assert np.array_equal(d, want), ("depth", s, lb, direction)
    check_tree(off, col, s, d, pred.cpu().numpy())
    return depth, pred, info


# ------------------------------------------------------------------------------------------------ golden graphs
@pytest.fixture(scope="module")
def golden_graphs(golden):
    out = {}
    for name, g in golden.items():
        csr = _csr(g["offsets"], g["indices"], g["values"], name, True)
        odd = gg.CSR(csr.n, csr.m, csr.offsets, _misaligned(csr.indices), _misaligned(csr.values), name, True)
        out[name] = (ess.Graph(csr), ess.Graph(odd), csr.host())
    return out


@pytest.mark.parametrize("lb", LBS)
def test_golden_trees(ctx, golden, golden_graphs, lb):
    """chesapeake, rmat_s10 and grid_24x17 from every golden source, forward and direction-optimised: depths equal to
    the golden vectors and to ess.bfs, parents valid."""
    for name, (g, _, (off, col, _)) in golden_graphs.items():
        for s in golden[name]["sources"]:
            s = int(s)
            want = golden[name][f"bfs_{s}"]
            for direction in ("forward", "optimized"):
                plain, _ = ess.bfs(ctx, g, s, lb=lb, direction=direction)
                assert np.array_equal(plain.cpu().numpy(), want), (name, s, lb, direction)
                _run_and_check(ctx, g, off, col, s, want, lb, direction)


def test_trees_on_a_misaligned_graph(ctx, golden, golden_graphs):
    """Column indices 4 bytes past a 16-byte boundary: advance drops to the scalar kernels by itself."""
    for name, (_, g, (off, col, _)) in golden_graphs.items():
        for s in golden[name]["sources"]:
            s = int(s)
            want = golden[name][f"bfs_{s}"]
            for lb in LBS:
                _run_and_check(ctx, g, off, col, s, want, lb, "forward")
            _run_and_check(ctx, g, off, col, s, want, "merge_path", "optimized")


# ------------------------------------------------------------------------------------------------ RMAT scale 16
@pytest.fixture(scope="module")
def s16():
    csr = gg.rmat_csr(16, device="cuda")
    return csr, ess.Graph(csr), csr.host()


@pytest.mark.parametrize("lb", LBS)
def test_rmat16_trees(ctx, s16, lb):
    """Every balancer, both directions. The optimised runs must go bottom-up and adopt vertices there, so the parents
    the pull kernels record are certainly checked."""
    csr, g, (off, col, _) = s16
    for s in [0] + gg.pick_sources(csr, 3):
        want = oracle.bfs(off, col, s)
        for direction in ("forward", "optimized"):
            _, _, info = _run_and_check(ctx, g, off, col, s, want, lb, direction)
            if direction == "optimized":
                assert info["pull_steps"] >= 1 and info["pull_found"] > 0, (s, lb, info)


FALLBACKS = [("pull_hints", 0), ("advance_engine", 0)]


@pytest.mark.parametrize("name,value", FALLBACKS)
def test_trees_on_the_fallback_kernels(ctx, s16, name, value):
    """Bottom-up without hints and the scalar advance kernels: RMAT scale 16 and arbitrary directed multigraphs."""
    csr, g, (off, col, _) = s16
    rng = np.random.default_rng(31)
    with knob(name, value):
        for s in [0] + gg.pick_sources(csr, 2):
            want = oracle.bfs(off, col, s)
            for lb in ("merge_path", "block_mapped"):
                _, _, info = _run_and_check(ctx, g, off, col, s, want, lb, "optimized")
                assert info["pull_steps"] >= 1 and info["pull_found"] > 0, (name, s, lb)
            _run_and_check(ctx, g, off, col, s, want, "thread_mapped", "forward")
        for trial in range(20):
            small = _arbitrary_multigraph(rng)
            o, c, _ = small.host()
            gs = ess.Graph(small, csc=ess.transpose(small))
            for s in {0, int(rng.integers(0, small.n))}:
                _run_and_check(ctx, gs, o, c, s, oracle.bfs(o, c, s), "merge_path", "optimized")


# ------------------------------------------------------------------------------------------------ other graph inputs
def test_trees_on_arbitrary_multigraphs(ctx):
    """Self loops, parallel edges, isolated vertices; the CSC is ess.transpose of the CSR. Parents must be tails of
    out-edges of the CSR."""
    rng = np.random.default_rng(32)
    for trial in range(30):
        small = _arbitrary_multigraph(rng)
        o, c, _ = small.host()
        gs = ess.Graph(small, csc=ess.transpose(small))
        for s in {0, int(rng.integers(0, small.n)), small.n - 1}:
            want = oracle.bfs(o, c, s)
            for lb in LBS:
                _run_and_check(ctx, gs, o, c, s, want, lb, "forward")
            _run_and_check(ctx, gs, o, c, s, want, "merge_path", "optimized")


def test_trees_with_int64_offsets_and_from_host(ctx):
    """A graph with 64-bit row offsets, and graphs built by Graph.from_host (the handle owns the device copies)."""
    csr = gg.rmat_csr(14, device="cuda")
    wide = gg.rmat_csr(14, device="cuda", offset_bits=64)
    assert wide.offsets.dtype == torch.int64 and torch.equal(wide.offsets, csr.offsets.long())
    off, col, _ = csr.host()
    graphs = {"int64 offsets": ess.Graph(wide), "from_host": ess.Graph.from_host(ctx, csr.pinned()),
              "from_host int64": ess.Graph.from_host(ctx, wide.pinned())}
    for s in [0] + gg.pick_sources(csr, 2):
        want = oracle.bfs(off, col, s)
        for what, g in graphs.items():
            for lb in LBS:
                for direction in ("forward", "optimized"):
                    _run_and_check(ctx, g, off, col, s, want, lb, direction)
    for g in graphs.values():
        g.close()


def test_isolated_source(ctx, s16):
    """A source without edges: pred[s] == s and every other entry -1."""
    csr, g, (off, col, _) = s16
    iso = int(np.flatnonzero(np.diff(off) == 0)[0])
    for lb in LBS:
        for direction in ("forward", "optimized"):
            depth, pred, _ = ess.bfs_tree(ctx, g, iso, lb=lb, direction=direction)
            want = np.full(csr.n, -1, np.int32)
            want[iso] = iso
            assert np.array_equal(pred.cpu().numpy(), want), (lb, direction)
            assert int(depth[iso]) == 0 and int((depth == INT32_MAX).sum()) == csr.n - 1


# ------------------------------------------------------------------------------------------------ caller buffers
def test_caller_buffers(ctx, s16):
    """pred_out full of random garbage (negative ids, ids past n, the source's id), a view 4 bytes past a 16-byte
    boundary, and one buffer pair reused across sources: the result never depends on what the buffer held."""
    csr, g, (off, col, _) = s16
    sources = [0] + gg.pick_sources(csr, 3)
    gen = torch.Generator(device="cuda").manual_seed(5)
    for direction in ("forward", "optimized"):
        for s in sources:
            want = oracle.bfs(off, col, s)
            garbage = torch.randint(-2**31, 2**31 - 1, (csr.n,), dtype=torch.int32, device="cuda", generator=gen)
            garbage[::7] = s
            depth, pred, _ = _run_and_check(ctx, g, off, col, s, want, "merge_path", direction, pred_out=garbage)
            assert pred.data_ptr() == garbage.data_ptr()
            odd = _misaligned(torch.full((csr.n,), 12345, dtype=torch.int32, device="cuda"))
            odd_depth = _misaligned(torch.zeros(csr.n, dtype=torch.int32, device="cuda"))
            _, pred, _ = _run_and_check(ctx, g, off, col, s, want, "bucketing", direction, out=odd_depth, pred_out=odd)
            assert pred.data_ptr() == odd.data_ptr()
        depth = torch.empty(csr.n, dtype=torch.int32, device="cuda")
        pred = torch.empty(csr.n, dtype=torch.int32, device="cuda")
        for lb in LBS:
            for s in sources + [int(np.flatnonzero(np.diff(off) == 0)[0])]:
                d, p, _ = _run_and_check(ctx, g, off, col, s, oracle.bfs(off, col, s), lb, direction, out=depth,
                                         pred_out=pred)
                assert d.data_ptr() == depth.data_ptr() and p.data_ptr() == pred.data_ptr()


def test_errors_are_raised_before_any_launch(ctx, s16):
    csr, g, _ = s16
    n = csr.n
    depth = torch.empty(n, dtype=torch.int32, device="cuda")
    bad = {
        "source -1": dict(source=-1),
        "source n": dict(source=n),
        "pred_out is out": dict(out=depth, pred_out=depth),
        "pred_out overlaps out": dict(out=depth, pred_out=torch.empty(2 * n, dtype=torch.int32, device="cuda")),
        "int64 pred_out": dict(pred_out=torch.empty(n, dtype=torch.int64, device="cuda")),
        "short pred_out": dict(pred_out=torch.empty(n - 1, dtype=torch.int32, device="cuda")),
        "host pred_out": dict(pred_out=torch.empty(n, dtype=torch.int32)),
        "strided pred_out": dict(pred_out=torch.empty(2 * n, dtype=torch.int32, device="cuda")[::2]),
    }
    bad["pred_out overlaps out"]["out"] = bad["pred_out overlaps out"]["pred_out"][n // 2: n // 2 + n]
    for what, kw in bad.items():
        s = kw.pop("source", 0)
        launches = ctx.launches()
        with pytest.raises(ess.EssentialsError):
            ess.bfs_tree(ctx, g, s, lb="merge_path", **kw)
        assert ctx.launches() == launches, what
    # direction-optimised needs the in-edges: a directed graph given as CSR only has none
    directed = gg.rmat_csr(10, symmetric=False, device="cuda")
    csr_only = ess.Graph(directed)
    with pytest.raises(ess.EssentialsError, match="CSC"):
        ess.bfs_tree(ctx, csr_only, 0, lb="merge_path", direction="optimized")
    # the C ABI's own checks (the binding stops these before the call)
    from ctypes import byref, c_void_p
    info = ess.RunInfo()
    L = ess.lib()
    p = c_void_p(depth.data_ptr())
    assert L.ess_bfs_tree(ctx.handle, g.handle, 0, p, None, 4, 0, 0.0, 0.0, byref(info)) != 0
    assert b"null" in L.ess_last_error()
    assert L.ess_bfs_tree(ctx.handle, g.handle, 0, p, p, 4, 0, 0.0, 0.0, byref(info)) != 0
    assert b"alias" in L.ess_last_error()
    assert L.ess_bfs_tree(ctx.handle, g.handle, n, p, c_void_p(depth.data_ptr() + 4), 4, 0, 0.0, 0.0,
                          byref(info)) != 0
    assert b"out of range" in L.ess_last_error()


def test_info_matches_ess_bfs(ctx, s16):
    """The tree run takes the same levels and the same push/pull decisions as the depth-only run."""
    csr, g, _ = s16
    s = gg.pick_sources(csr, 1)[0]
    for direction in ("forward", "optimized"):
        _, a = ess.bfs(ctx, g, s, lb="merge_path", direction=direction)
        _, _, b = ess.bfs_tree(ctx, g, s, lb="merge_path", direction=direction)
        for k in ("iterations", "pull_steps", "push_steps"):
            assert a[k] == b[k], (direction, k)


# ------------------------------------------------------------------------------------------------ RMAT scale 20
@pytest.fixture(scope="module")
def s20():
    csr = gg.rmat_csr(20, device="cuda")
    return csr, ess.Graph(csr)


@pytest.mark.parametrize("lb", LBS)
def test_rmat20_trees_on_the_device(ctx, s20, lb):
    """Scale 20, direction-optimised, checked on the device by the checker scripts/bfs_tree_cost.py uses (small
    chunks, so its chunked edge pass runs many times)."""
    csr, g = s20
    for s in gg.pick_sources(csr, 2):
        plain, _ = ess.bfs(ctx, g, s, lb=lb, direction="optimized")
        depth, pred, info = ess.bfs_tree(ctx, g, s, lb=lb, direction="optimized")
        assert torch.equal(plain, depth), (lb, s)
        assert info["pull_found"] > 0
        v = tree_violations(csr.offsets, csr.indices, s, depth, pred, chunk=1 << 22)
        assert not any(v.values()), (lb, s, v)


def test_device_checker_finds_each_broken_rule(ctx, s16):
    """tree_violations is the only check the cost measurement has: each rule it enforces must fire on a tree broken in
    exactly that way."""
    csr, g, _ = s16
    s = gg.pick_sources(csr, 1)[0]
    depth, pred, _ = ess.bfs_tree(ctx, g, s, lb="merge_path", direction="optimized")
    assert not any(tree_violations(csr.offsets, csr.indices, s, depth, pred, chunk=1 << 16).values())
    reached = (depth != INT32_MAX).nonzero().squeeze(1)
    v = int(reached[reached != s][-1])
    grand = int(pred[int(pred[v])]) if int(pred[v]) != s else None
    broken = {"source": (s, -1), "unreached": (v, -1), "range": (v, csr.n)}
    if grand is not None:
        broken["depth"] = (v, grand)
    off, col, _ = csr.host()
    nbrs = set(col[off[v]:off[v + 1]].tolist())
    same_level = (depth == depth[v] - 1).nonzero().squeeze(1).tolist()
    stranger = next(u for u in same_level if u not in nbrs)
    broken["edge"] = (v, stranger)
    for rule, (at, value) in broken.items():
        p = pred.clone()
        p[at] = value
        got = tree_violations(csr.offsets, csr.indices, s, depth, p, chunk=1 << 16)
        assert got[rule] > 0, (rule, got)
