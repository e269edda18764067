"""GPU suite (-m gpu): advance and filter against the buffers callers hand them.

The algorithm tests elsewhere run every operator on buffers the library sized itself. These tests hand the
operators what a caller may pass instead: output buffers of every capacity around the frontier's worst case
(Σdeg), graph arrays freed and rebuilt at the same address, and tensor views that start 4 bytes past a 16-byte
boundary. They also run the fallback kernels that only a knob or a misaligned graph selects: the scalar advance
kernels (advance_engine 0) and bottom-up without hints (pull_hints 0).
Every expected value comes from NumPy or the CPU oracle."""
import numpy as np
import pytest
import torch

import essentials_b200 as ess
import oracle
from essentials_b200 import graphgen as gg

pytestmark = pytest.mark.gpu

LBS = list(ess.IMPLEMENTED_LOAD_BALANCERS)
BIG_DEGREE = 4096  # kernels::big_degree: lists this long are expanded grid-wide (bucketing's third bin)
WARP_DEGREE = 32   # kernels::warp_degree: bucketing gives lists this long a warp
KNOB_DEFAULTS = {"advance_engine": 1, "pull_hints": 1, "sssp_fused_unique": 1}


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


def _expected_advance(off, col, frontier, modulus):
    kept, calls = [], np.zeros(max(col.size, 1), np.int64)
    for v in frontier:
        if v < 0:
            continue
        e = np.arange(off[v], off[v + 1], dtype=np.int64)
        calls[e] += 1
        keep = (v + col[e].astype(np.int64) + e) % modulus != 0
        kept.append(col[e][keep])
    return (np.sort(np.concatenate(kept)) if kept else np.zeros(0, np.int32)), calls


def _is_sub_multiset(part, whole):
    pv, pc = np.unique(part, return_counts=True)
    wv, wc = np.unique(whole, return_counts=True)
    if pv.size == 0 or wv.size == 0:
        return pv.size == 0
    at = np.minimum(np.searchsorted(wv, pv), wv.size - 1)
    return bool(np.all(wv[at] == pv) and np.all(pc <= wc[at]))


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


# ------------------------------------------------------------------------------------------------ A. output capacity
@pytest.fixture(scope="module")
def buffer_graph():
    """Directed multigraph built for the capacity tests. Out-edges: vertex 0 is a hub of degree 4500 (>= BIG_DEGREE),
    vertices 2..201 have 33..800 edges (bucketing's warp bin), 202..4201 have 2..31 (its thread bin), the rest none.
    In-edges: vertex 1 is the hub of the CSC view (4200 in-edges), vertices 5990.. have none."""
    rng = np.random.default_rng(11)
    n, reach = 6000, 5990
    mids, leaves = np.arange(2, 202), np.arange(202, 4202)
    deg = np.concatenate([rng.integers(32, 800, mids.size), rng.integers(1, 31, leaves.size)])
    src = np.concatenate([np.zeros(4500, np.int64), np.repeat(np.concatenate([mids, leaves]), deg),
                          np.concatenate([mids, leaves])])
    dst = np.concatenate([rng.choice(np.arange(2, reach), 4500, replace=False), rng.integers(0, reach, deg.sum()),
                          np.ones(mids.size + leaves.size, np.int64)])
    off, col, _ = _from_edges(n, src, dst)
    csr = _csr(off, col, None, "buffers", False)
    csc = ess.transpose(csr)
    g = ess.Graph(csr, csc=csc)
    views = {"forward": csr.host()[:2], "backward": csc.host()[:2]}
    for direction, (o, _) in views.items():
        d = np.diff(o)
        assert d.max() >= BIG_DEGREE and ((d >= WARP_DEGREE) & (d < BIG_DEGREE)).any()
        assert ((d > 0) & (d < WARP_DEGREE)).any() and (d == 0).any(), direction
    frontiers = {}
    for direction, (o, c) in views.items():
        d = np.diff(o)
        hub = int(np.argmax(d))

        def noisy(items, holes, dups):
            f = np.concatenate([items, -np.ones(holes, np.int64), items[:dups]])
            rng.shuffle(f)
            return f.astype(np.int32)

        bins = [np.flatnonzero((d > 0) & (d < WARP_DEGREE)), np.flatnonzero((d >= WARP_DEGREE) & (d < BIG_DEGREE)),
                np.flatnonzero(d == 0)]
        cases = {
            "512 items (single-launch merge path)": noisy(rng.integers(0, n, 480), 20, 12),
            "1024 items (scalar small-frontier limit)": noisy(rng.integers(0, n, 990), 20, 14),
            "8000 items": noisy(rng.integers(0, n, 7000), 300, 700),
            "hub repeated past m": np.full(int(d.sum()) // int(d[hub]) + 2, hub, np.int32),
            "every degree bin": noisy(np.concatenate([[hub], rng.choice(bins[0], 200), rng.choice(bins[1], 40),
                                                      rng.choice(bins[2], 20)]), 10, 30),
        }
        assert cases["512 items (single-launch merge path)"].size == 512
        assert cases["1024 items (scalar small-frontier limit)"].size == 1024
        assert int(d[cases["hub repeated past m"]].sum()) > c.size
        for label, f in cases.items():
            want, want_calls = _expected_advance(o, c, f, 3)
            frontiers[direction, label] = (f, int(d[f[f >= 0]].sum()), want, want_calls[: c.size])
    return g, frontiers


def _capacities(worst, produced):
    """1, Σdeg - 1, Σdeg, Σdeg + 1 (what the capacity guard compares), and one less than the output itself."""
    return sorted({c for c in (1, worst - 1, worst, worst + 1, produced - 1) if c >= 1})


def _check_probe(run, want, want_calls, cap, unique, what):
    """Runs one probe at capacity `cap` and checks the produced count, the output and the per-edge call counts."""
    try:
        out, calls = run()
        got = np.sort(out.cpu().numpy())
        assert got.size == want.size, (what, "count", got.size, want.size)
        assert np.array_equal(got, want), (what, "output")
    except ess.OutputOverflow as e:
        assert want.size > cap, (what, "overflow reported for an output that fits", e.produced)
        assert e.produced == want.size, (what, "produced count", e.produced, want.size)
        prefix = e.prefix.cpu().numpy()
        assert prefix.size == cap, what
        assert _is_sub_multiset(prefix, want), (what, "prefix is not part of the output")
        if unique:
            assert np.unique(prefix).size == prefix.size, (what, "duplicate in a unique output")
        calls = e.calls
    assert np.array_equal(calls.cpu().numpy()[: want_calls.size], (2 if unique else 1) * want_calls), \
        (what, "operator calls per edge")


@pytest.mark.parametrize("engine", [1, 0])
@pytest.mark.parametrize("lb", LBS)
def test_advance_output_capacity(ctx, buffer_graph, lb, engine):
    """operators::advance::execute and execute_unique into caller buffers from 1 element to Σdeg + 1. A buffer
    smaller than Σdeg takes the overflow path: nothing runs, the operator grows the output and relaunches, so the
    operator still runs exactly once per (item, edge) (twice for the unique probe, which calls it twice). Only when
    the kept neighbours themselves do not fit is the overflow reported, with the full count."""
    g, frontiers = buffer_graph
    with knob("advance_engine", engine):
        for (direction, label), (f, worst, want, want_calls) in frontiers.items():
            ft = torch.from_numpy(f).cuda()
            for cap in _capacities(worst, want.size):
                _check_probe(lambda: ess.advance_probe(ctx, g, ft, lb=lb, direction=direction, capacity=cap),
                             want, want_calls, cap, False, (lb, engine, direction, label, cap))
            if direction == "forward":
                uniq = np.unique(want)
                for cap in _capacities(worst, uniq.size):
                    _check_probe(lambda: ess.advance_unique_probe(ctx, g, ft, lb=lb, capacity=cap),
                                 uniq, want_calls, cap, True, (lb, engine, "unique", label, cap))
            out, _ = ess.advance_probe(ctx, g, ft, lb=lb, direction=direction)  # default buffer: never truncates
            assert out.numel() == want.size, (lb, engine, direction, label)


# ------------------------------------------------------------------------------------------------ B. graph lifetimes
def _ring(n):
    return np.arange(n + 1, dtype=np.int64), (np.arange(n) + 1) % n


def _star(n):
    """Vertex 0 -> every other vertex: offsets [0, n-1, n-1, ...]."""
    off = np.full(n + 1, n - 1, np.int64)
    off[0] = 0
    return off, np.arange(1, n)


def _hub_probes(ctx, g, off, col, what):
    """The repeated-hub probe of part A with the thread- and block-mapped balancers, whose output guard trusts the
    cached max degree: by default, and with a buffer one element short of the output."""
    hub = int(np.argmax(np.diff(off)))
    f = np.full(col.size // int(off[hub + 1] - off[hub]) + 2, hub, np.int32)
    want, want_calls = _expected_advance(off, col, f, 3)
    ft = torch.from_numpy(f).cuda()
    for lb in ("thread_mapped", "block_mapped"):
        out, calls = ess.advance_probe(ctx, g, ft, lb=lb)
        assert out.numel() == want.size, (what, lb, "count", out.numel(), want.size)
        assert np.array_equal(np.sort(out.cpu().numpy()), want), (what, lb)
        assert np.array_equal(calls.cpu().numpy()[: col.size], want_calls[: col.size]), (what, lb)
        cap = want.size - 1
        _check_probe(lambda: ess.advance_probe(ctx, g, ft, lb=lb, capacity=cap), want, want_calls[: col.size], cap,
                     False, (what, lb, cap))


def test_max_degree_cache_follows_the_graph_not_its_address():
    """The thread- and block-mapped advances skip their Σdeg pass when nf * max_degree fits the output, and the max
    degree is cached per context. A graph built over memory a freed graph used (same offsets address, same n) must
    not inherit the old graph's value: (a) caller arrays rewritten in place, (b) the handle's own pool blocks through
    Graph.from_host, (c) two live graphs used alternately."""
    c = ess.Context(0)
    n = 6000
    # (a) one offsets tensor, first a ring (max degree 1), then a star (max degree n - 1)
    ring_off, ring_col = _ring(n)
    T = torch.from_numpy(ring_off.astype(np.int32)).cuda()
    a = ess.Graph(gg.CSR(n, n, T, torch.from_numpy(ring_col.astype(np.int32)).cuda(), None, "ring", False))
    out, _ = ess.advance_probe(c, a, torch.arange(n, dtype=torch.int32, device="cuda"), lb="block_mapped")
    assert out.numel() == np.count_nonzero((np.arange(n) + ring_col + np.arange(n)) % 3)
    a.close()
    star_off, star_col = _star(n)
    T.copy_(torch.from_numpy(star_off.astype(np.int32)))
    b = ess.Graph(gg.CSR(n, n - 1, T, torch.from_numpy(star_col.astype(np.int32)).cuda(), None, "star", False))
    _hub_probes(c, b, star_off, star_col, "(a) rewritten in place")
    b.close()

    # (b) the same swap through Graph.from_host: the handle's device pool hands the ring's blocks to the star
    def host_graph(off, col):
        rng = np.random.default_rng(3)
        src = np.repeat(np.arange(n), np.diff(off))
        both = np.concatenate([src, col]), np.concatenate([col, src])  # symmetric: hints and a CSC view
        key = np.unique(both[0] * n + both[1])
        s, d = key // n, key % n
        w = rng.choice(np.array([0.5, 1.0, 2.25, 7.0], np.float32), s.size)
        w = np.maximum(w, w[np.searchsorted(key, d * n + s)])  # same weight both ways
        o, cl, wv = _from_edges(n, s, d, w)
        return o, cl, wv, ess.Graph.from_host(c, _csr(o, cl, wv, "host", True, device="cpu"))

    o, cl, wv, a = host_graph(*_ring(n))
    ess.advance_probe(c, a, torch.arange(n, dtype=torch.int32, device="cuda"), lb="block_mapped")
    a.close()
    o, cl, wv, b = host_graph(*_star(n))
    for s in (0, 1, n - 1):
        want = oracle.bfs(o, cl, s)
        for lb in ("thread_mapped", "block_mapped"):
            d, _ = ess.bfs(c, b, s, lb=lb)
            assert np.array_equal(d.cpu().numpy(), want), ("(b) bfs", s, lb)
        d, _ = ess.bfs(c, b, s, lb="merge_path", direction="optimized")
        assert np.array_equal(d.cpu().numpy(), want), ("(b) bfs optimized", s)
        with knob("sssp_fused_unique", 0):  # advance + bypass filter: the output frontier repeats vertices
            for lb in ("thread_mapped", "block_mapped"):
                d, _ = ess.sssp(c, b, s, lb=lb)
                assert np.array_equal(d.cpu().numpy(), oracle.sssp(o, cl, wv, s)), ("(b) sssp", s, lb)
    _hub_probes(c, b, o, cl, "(b) from_host")
    b.close()

    # (c) two live graphs, same n, max degrees 1 and n - 1, used alternately on one context
    ring = ess.Graph(_csr(*_ring(n), None, "ring", False))
    star = ess.Graph(_csr(*_star(n), None, "star", False))
    for turn in range(4):
        if turn % 2:
            _hub_probes(c, star, *_star(n), f"(c) star, turn {turn}")
        else:
            _hub_probes(c, ring, *_ring(n), f"(c) ring, turn {turn}")
    c.close()


# ------------------------------------------------------------------------------------------------ C. misaligned views
@pytest.fixture(scope="module")
def golden_graphs(golden):
    out = {}
    for name, g in golden.items():
        csr = _csr(g["offsets"], g["indices"], g["values"], name, True)
        odd = gg.CSR(csr.n, csr.m, csr.offsets, _misaligned(csr.indices), _misaligned(csr.values), name, True)
        out[name] = (ess.Graph(csr), ess.Graph(odd), odd)
    return out


@pytest.mark.parametrize("engine", [1, 0])
def test_advance_on_a_misaligned_frontier(ctx, buffer_graph, engine):
    """The merge-path preparation passes read the frontier 128 bits at a time; a frontier view at a 4-byte offset
    must take their scalar path. 3000 items: past the single-launch limits, so the preparation passes run."""
    g, frontiers = buffer_graph
    rng = np.random.default_rng(8)
    f = rng.integers(0, g.n, 3000).astype(np.int32)
    f[rng.random(f.size) < 0.05] = -1
    ft = _misaligned(torch.from_numpy(f).cuda())
    with knob("advance_engine", engine):
        for direction, view in (("forward", g.csr), ("backward", g.csc)):
            off, col, _ = view.host()
            want, want_calls = _expected_advance(off, col, f, 3)
            for lb in LBS:
                out, calls = ess.advance_probe(ctx, g, ft, lb=lb, direction=direction)
                assert np.array_equal(np.sort(out.cpu().numpy()), want), (lb, engine, direction)
                assert np.array_equal(calls.cpu().numpy()[: col.size], want_calls[: col.size]), (lb, engine, direction)
                if direction == "forward":
                    out, calls = ess.advance_unique_probe(ctx, g, ft, lb=lb)
                    assert np.array_equal(np.sort(out.cpu().numpy()), np.unique(want)), (lb, engine, "unique")
                    assert np.array_equal(calls.cpu().numpy()[: col.size], 2 * want_calls[: col.size])


@pytest.mark.parametrize("alg", ["predicated", "remove", "compact", "bypass"])
def test_filter_on_misaligned_items(ctx, golden_graphs, alg):
    """filter loads its input 128 bits at a time, and bypass also stores that way: both on views at a 4-byte offset,
    bypass in place on one."""
    g = golden_graphs["rmat_s10"][0]
    rng = np.random.default_rng(10)
    for size in (3, 4, 5, 1023, 1025, 40000):
        items = rng.integers(0, g.n, size).astype(np.int32)
        items[rng.random(size) < 0.1] = -1
        keep = (items >= 0) & (items % 3 != 0)
        out, calls = ess.filter_probe(ctx, g, _misaligned(torch.from_numpy(items).cuda()), alg=alg, modulus=3)
        want = np.where(keep, items, -1) if alg == "bypass" else items[keep]
        assert np.array_equal(out.cpu().numpy(), want), (alg, size)
        assert np.array_equal(calls.cpu().numpy()[: g.n], np.bincount(items[items >= 0], minlength=g.n)), (alg, size)
        if alg == "bypass":
            view = _misaligned(torch.from_numpy(items).cuda())
            out, _ = ess.filter_probe(ctx, g, view, alg="bypass", modulus=3, in_place=True)
            assert out.data_ptr() == view.data_ptr()
            assert np.array_equal(view.cpu().numpy(), want), ("in place", size)


def test_sssp_into_misaligned_outputs(ctx, golden, golden_graphs):
    """run_delta reads the distances 128 bits at a time; the distance array is the caller's `out`."""
    for name, (g, _, _) in golden_graphs.items():
        for s in golden[name]["sources"]:
            want = golden[name][f"sssp_{s}"]
            runs = {"delta": lambda o: ess.sssp_delta(ctx, g, int(s), out=o),
                    "delta 3e38": lambda o: ess.sssp_delta(ctx, g, int(s), delta=3e38, out=o),
                    "near_far": lambda o: ess.sssp_near_far(ctx, g, int(s), out=o),
                    "block_mapped": lambda o: ess.sssp(ctx, g, int(s), lb="block_mapped", out=o),
                    "merge_path": lambda o: ess.sssp(ctx, g, int(s), lb="merge_path", out=o)}
            for what, run in runs.items():
                out = _misaligned(torch.zeros(g.n, dtype=torch.float32, device="cuda"))
                dist, _ = run(out)
                assert dist.data_ptr() == out.data_ptr()
                assert np.array_equal(out.cpu().numpy(), want), (name, int(s), what)


def test_traversals_on_misaligned_graph_arrays(ctx, golden, golden_graphs):
    """A graph whose column indices and weights start 4 bytes past a 16-byte boundary cannot use the 128-bit quad
    engine: advance falls back to the scalar kernels by itself (advance_engine stays 1). Every traversal must still
    match the golden vectors and the oracle."""
    for name, (_, g, odd) in golden_graphs.items():
        off, col, val = odd.host()
        for s in golden[name]["sources"]:
            s = int(s)
            want_bfs, want_sssp = golden[name][f"bfs_{s}"], golden[name][f"sssp_{s}"]
            assert np.array_equal(want_bfs, oracle.bfs(off, col, s))
            assert np.array_equal(want_sssp, oracle.sssp(off, col, val, s))
            for lb in LBS:
                d, _ = ess.bfs(ctx, g, s, lb=lb)
                assert np.array_equal(d.cpu().numpy(), want_bfs), (name, s, "bfs", lb)
                d, _ = ess.sssp(ctx, g, s, lb=lb)
                assert np.array_equal(d.cpu().numpy(), want_sssp), (name, s, "sssp", lb)
            d, _ = ess.bfs(ctx, g, s, lb="merge_path", direction="optimized")
            assert np.array_equal(d.cpu().numpy(), want_bfs), (name, s, "bfs optimized")
            d, _ = ess.sssp_delta(ctx, g, s)
            assert np.array_equal(d.cpu().numpy(), want_sssp), (name, s, "delta")
            d, _ = ess.sssp_near_far(ctx, g, s)
            assert np.array_equal(d.cpu().numpy(), want_sssp), (name, s, "near_far")


# ------------------------------------------------------------------------------------------------ D. fallback kernels
def _arbitrary_multigraph(rng):
    """Small directed multigraph with self loops, parallel edges, isolated vertices, zero and tied weights."""
    n = int(rng.integers(2, 70))
    m = int(rng.integers(1, 400))
    src, dst = rng.integers(0, n, m), rng.integers(0, n, m)
    w = rng.choice(np.array([0.0, 0.5, 1.0, 1.0, 2.25, 7.0, 63.984375], np.float32), m)
    off, col, val = _from_edges(n, src, dst, w)
    return _csr(off, col, val, "arbitrary", False)


FALLBACKS = [("pull_hints", 0), ("advance_engine", 0)]


@pytest.fixture(scope="module")
def s16():
    csr = gg.rmat_csr(16, device="cuda")
    return csr, ess.Graph(csr), csr.host()


@pytest.mark.parametrize("name,value", FALLBACKS)
def test_optimized_bfs_fallbacks(ctx, s16, name, value):
    """Direction-optimised BFS without the bottom-up hints and with the scalar advance kernels: bit-equal to the oracle on RMAT scale 16 (which must switch to bottom-up) and on arbitrary
    directed multigraphs (CSR + transposed CSC)."""
    csr, g, (off, col, _) = s16
    rng = np.random.default_rng(21)
    with knob(name, value):
        for s in [0] + gg.pick_sources(csr, 2):
            for lb in ("merge_path", "block_mapped"):
                depth, info = ess.bfs(ctx, g, s, lb=lb, direction="optimized")
                assert np.array_equal(depth.cpu().numpy(), oracle.bfs(off, col, s)), (name, s, lb)
                assert info["pull_steps"] >= 1, "a Kronecker graph must trigger the bottom-up switch"
        for trial in range(20):
            small = _arbitrary_multigraph(rng)
            o, c, _ = small.host()
            gs = ess.Graph(small, csc=ess.transpose(small))
            for s in {0, int(rng.integers(0, small.n))}:
                d, _ = ess.bfs(ctx, gs, s, lb="merge_path", direction="optimized")
                assert np.array_equal(d.cpu().numpy(), oracle.bfs(o, c, s)), (name, trial, s)


def test_sssp_on_the_scalar_advance_kernels(ctx, golden, golden_graphs):
    """SSSP as frontier recipe (fused advance + uniquify, and the reference's advance + bypass pair) and as dense delta
    stepping, all on the scalar advance kernels: bit-equal to the golden vectors and, on arbitrary multigraphs, to the
    oracle."""
    rng = np.random.default_rng(22)
    smalls = [_arbitrary_multigraph(rng) for _ in range(15)]
    with knob("advance_engine", 0):
        for fused in (1, 0):
            with knob("sssp_fused_unique", fused):
                for name, (g, _, _) in golden_graphs.items():
                    for s in golden[name]["sources"]:
                        for lb in LBS:
                            d, _ = ess.sssp(ctx, g, int(s), lb=lb)
                            assert np.array_equal(d.cpu().numpy(), golden[name][f"sssp_{s}"]), (name, s, lb, fused)
                for small in smalls:
                    o, c, w = small.host()
                    d, _ = ess.sssp(ctx, ess.Graph(small), 0, lb="merge_path")
                    assert np.array_equal(d.cpu().numpy(), oracle.sssp(o, c, w, 0)), ("arbitrary", fused)
        for name, (g, _, _) in golden_graphs.items():
            for s in golden[name]["sources"]:
                d, _ = ess.sssp_delta(ctx, g, int(s))
                assert np.array_equal(d.cpu().numpy(), golden[name][f"sssp_{s}"]), (name, s, "delta")
        for small in smalls:
            o, c, w = small.host()
            d, _ = ess.sssp_delta(ctx, ess.Graph(small), 0, delta=1.0)
            assert np.array_equal(d.cpu().numpy(), oracle.sssp(o, c, w, 0)), ("arbitrary", "delta")
