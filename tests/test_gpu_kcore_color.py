"""GPU suite (-m gpu): k-core and colouring on every path they run, the random stream colouring draws from, and the
`out=` buffers of the entry points that write one label per vertex.

k-core runs, per inner round, one advance (the peel), a parallel_for and a predicated filter whose op is an atomic
decrement. So it is run here through every advance kernel: the grid-wide hub kernel (rows of >= 4096 edges), bucketing's
warp and thread bins, the scalar kernels (advance_engine 0, or a misaligned graph), 64-bit offsets and graphs built
from host arrays. The inputs have self-loops, parallel edges and isolated vertices, some are directed, and some peels
are thousands of inner rounds deep. Colouring is run on graphs where adjacent vertices draw the same random value, so
both branches of its vertex-id tie-break decide colours. Every expected value comes from the CPU oracle or from a
closed form, and every comparison of core numbers, colours and random values is bit for bit."""
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
KNOB_DEFAULTS = {"advance_engine": 1}
SENTINEL = -559038737  # 0xDEADBEEF as int32: what a caller's buffer holds where the library must not write


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


def _from_edges(n, src, dst):
    """Offsets (int64) and column indices of the directed edge list, rows sorted by destination."""
    src, dst = np.asarray(src, np.int64), np.asarray(dst, np.int64)
    order = np.lexsort((dst, src))
    off = np.zeros(n + 1, np.int64)
    np.add.at(off, src + 1, 1)
    return np.cumsum(off), dst[order].astype(np.int32)


def _symmetric(n, u, v):
    """Both directions of every undirected edge (u, v); a self-loop is stored once."""
    u, v = np.asarray(u, np.int64), np.asarray(v, np.int64)
    loop = u == v
    return _from_edges(n, np.concatenate([u, v[~loop]]), np.concatenate([v, u[~loop]]))


def _csr(off, col, name, symmetric, wide=False, device="cuda"):
    return gg.CSR(off.size - 1, col.size, torch.from_numpy(off.astype(np.int64 if wide else np.int32)).to(device),
                  torch.from_numpy(col.astype(np.int32)).to(device), None, name, symmetric)


def _misaligned(t):
    """Copy of `t` in a view one element into a fresh buffer: 4 bytes past a 16-byte boundary for 4-byte types."""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    view = buf[1:]
    view.copy_(t)
    assert view.data_ptr() % 16 == 4
    return view


def _arbitrary_multigraph(rng):
    """Small directed multigraph with self loops, parallel edges and isolated vertices."""
    n = int(rng.integers(2, 70))
    m = int(rng.integers(1, 400))
    off, col = _from_edges(n, rng.integers(0, n, m), rng.integers(0, n, m))
    return _csr(off, col, "arbitrary", False)


def _bins(off):
    d = np.diff(off)
    return {"hub": int((d >= BIG_DEGREE).sum()), "warp": int(((d >= WARP_DEGREE) & (d < BIG_DEGREE)).sum()),
            "thread": int(((d > 0) & (d < WARP_DEGREE)).sum()), "isolated": int((d == 0).sum())}


# ------------------------------------------------------------------------------------------------ graphs
@pytest.fixture(scope="module")
def multigraph():
    """Symmetric multigraph that reaches every advance bin: vertex 0 is a hub of 4600 distinct neighbours plus parallel
    edges, vertices 4601..4800 have 40..700 random partners (bucketing's warp bin), 4801..10999 have 1..3 (its thread
    bin), 11000..11999 are isolated; 300 self-loops and 600 doubled edges are spread over the rest."""
    rng = np.random.default_rng(31)
    n, reach = 12000, 11000
    hub_nbrs, mids, small = np.arange(1, 4601), np.arange(4601, 4801), np.arange(4801, reach)
    mid_deg, small_deg = rng.integers(40, 700, mids.size), rng.integers(1, 4, small.size)
    u = np.concatenate([np.zeros(hub_nbrs.size, np.int64), np.repeat(mids, mid_deg), np.repeat(small, small_deg)])
    v = np.concatenate([hub_nbrs, rng.integers(1, reach, mid_deg.sum() + small_deg.sum())])
    keep = u != v
    u, v = u[keep], v[keep]
    twice = rng.choice(u.size, 600, replace=False)
    twice[:40] = rng.choice(hub_nbrs.size, 40, replace=False)  # parallel edges at the hub too
    loops = rng.choice(np.arange(1, reach), 300, replace=False)
    off, col = _symmetric(n, np.concatenate([u, u[twice], loops]), np.concatenate([v, v[twice], loops]))
    bins = _bins(off)
    assert all(bins.values()), bins
    assert np.diff(off)[0] >= BIG_DEGREE + 500
    rows = np.repeat(np.arange(n), np.diff(off))
    assert int((rows == col).sum()) == loops.size, "self-loops"
    assert np.unique(rows * n + col).size < col.size, "parallel edges"
    want = oracle.kcore(off, col)
    assert want.max() >= 8 and np.unique(want).size >= 6, "a peel of several levels"
    csr = _csr(off, col, "multigraph", True)
    return csr, ess.Graph(csr), off, col, want


@pytest.fixture(scope="module")
def s16():
    csr = gg.rmat_csr(16, device="cuda")
    return csr, ess.Graph(csr), csr.host()


@pytest.fixture(scope="module")
def s18():
    csr = gg.rmat_csr(18, device="cuda")
    return csr, ess.Graph(csr), csr.host()


@pytest.fixture(scope="module")
def deep_peel():
    """Components whose core numbers are known in closed form, under a random relabelling of the vertex ids:
    K_64 (core 63: 63 levels); a 3000-vertex path (core 1, peeled two vertices per inner round: ~1500 rounds of
    2-vertex frontiers at k = 1); a 777-cycle (core 2); a star of 5000 leaves whose centre also lies on a triangle (the
    centre's degree falls from 5002 to 2 in one filter at k = 1 and must not enter that level: core 2); a star of 4000
    leaves whose centre is tied to one vertex of a K_5 (its degree falls from 4001 to 1 in one filter, crossing k + 1 = 2
    exactly there: core 1, the K_5 core 4); 100 isolated vertices (core 0)."""
    edges, want = [], []

    def block(size, core):
        first = len(want)
        want.extend([core] * size)
        return first

    k64 = block(64, 63)
    a, b = np.triu_indices(64, 1)
    edges.append((k64 + a, k64 + b))
    path = block(3000, 1)
    edges.append((path + np.arange(2999), path + np.arange(1, 3000)))
    cyc = block(777, 2)
    edges.append((cyc + np.arange(777), cyc + (np.arange(777) + 1) % 777))
    centre = block(3, 2)  # centre, and the two other triangle vertices
    leaves = block(5000, 1)
    edges.append((np.full(5000, centre), leaves + np.arange(5000)))
    edges.append((centre + np.array([0, 0, 1]), centre + np.array([1, 2, 2])))
    centre2 = block(1, 1)
    leaves2 = block(4000, 1)
    k5 = block(5, 4)
    edges.append((np.full(4000, centre2), leaves2 + np.arange(4000)))
    a, b = np.triu_indices(5, 1)
    edges.append((k5 + a, k5 + b))
    edges.append((np.array([centre2]), np.array([k5])))
    block(100, 0)
    n = len(want)
    perm = np.random.default_rng(5).permutation(n)
    u = perm[np.concatenate([e[0] for e in edges])]
    v = perm[np.concatenate([e[1] for e in edges])]
    closed = np.empty(n, np.int32)
    closed[perm] = np.array(want, np.int32)
    off, col = _symmetric(n, u, v)
    assert np.diff(off).max() >= BIG_DEGREE
    csr = _csr(off, col, "deep-peel", True)
    return csr, ess.Graph(csr), off, col, closed


# ------------------------------------------------------------------------------------------------ k-core
@pytest.mark.parametrize("engine", [1, 0])
@pytest.mark.parametrize("lb", LBS)
def test_kcore_every_advance_path(ctx, multigraph, lb, engine):
    """The peel's advance through the hub kernel, bucketing's warp and thread bins, and (engine 0) the scalar kernels,
    on self-loops, parallel edges and isolated vertices."""
    _, g, _, _, want = multigraph
    with knob("advance_engine", engine):
        k, _ = ess.kcore(ctx, g, lb=lb)
    assert np.array_equal(k.cpu().numpy(), want), (lb, engine)


@pytest.mark.parametrize("lb", LBS)
def test_kcore_rmat16(ctx, s16, lb):
    _, g, (off, col, _) = s16
    k, _ = ess.kcore(ctx, g, lb=lb)
    assert np.array_equal(k.cpu().numpy(), oracle.kcore(off, col)), lb


@pytest.mark.parametrize("lb", ["merge_path", "block_mapped"])
def test_kcore_rmat18(ctx, s18, lb):
    _, g, (off, col, _) = s18
    k, _ = ess.kcore(ctx, g, lb=lb)
    assert np.array_equal(k.cpu().numpy(), oracle.kcore(off, col)), lb


@pytest.mark.parametrize("lb", LBS)
def test_kcore_deep_peels(ctx, deep_peel, lb):
    """Thousands of inner rounds on tiny frontiers (merge path's single-launch kernel), 63 levels, and a degree that
    drops by thousands in one filter: the closed-form core numbers, which the oracle also gives."""
    _, g, off, col, closed = deep_peel
    assert np.array_equal(oracle.kcore(off, col), closed)
    k, _ = ess.kcore(ctx, g, lb=lb)
    assert np.array_equal(k.cpu().numpy(), closed), lb


def test_kcore_directed_multigraphs(ctx):
    """The reference's semantics on directed inputs: a vertex's degree is its out-degree (a self-loop counts once), and
    peeling it decrements its out-neighbours."""
    rng = np.random.default_rng(41)
    for trial in range(40):
        csr = _arbitrary_multigraph(rng)
        off, col, _ = csr.host()
        want = oracle.kcore(off, col)
        g = ess.Graph(csr)
        for engine in (1, 0):
            with knob("advance_engine", engine):
                for lb in LBS:
                    k, _ = ess.kcore(ctx, g, lb=lb)
                    assert np.array_equal(k.cpu().numpy(), want), (trial, lb, engine)


def _graph_form(ctx, csr, off, col, form):
    if form == "int64 offsets":
        return ess.Graph(_csr(off, col, csr.name, True, wide=True))
    if form == "misaligned indices":
        return ess.Graph(gg.CSR(csr.n, csr.m, csr.offsets, _misaligned(csr.indices), None, csr.name, True))
    wide = form.endswith("int64")
    host = _csr(off, col, csr.name, True, wide=wide, device="cpu")
    return ess.Graph.from_host(ctx, host.pinned() if "pinned" in form else host)


FORMS = ["int64 offsets", "misaligned indices", "host pinned", "host pageable", "host pinned int64",
         "host pageable int64"]


@pytest.mark.parametrize("form", FORMS)
def test_kcore_and_color_graph_forms(ctx, multigraph, form):
    """64-bit offsets, column indices 4 bytes past a 16-byte boundary (the scalar kernels) and graphs built from pinned
    or pageable host arrays: byte-equal to the 32-bit device graph and to the oracle."""
    csr, g, off, col, want = multigraph
    other = _graph_form(ctx, csr, off, col, form)
    assert other.offset_bits == (64 if "int64" in form else 32)
    for lb in LBS:
        plain, _ = ess.kcore(ctx, g, lb=lb)
        k, _ = ess.kcore(ctx, other, lb=lb)
        assert torch.equal(k, plain), (form, lb)
        assert np.array_equal(k.cpu().numpy(), want), (form, lb)
    plain, pi = ess.color(ctx, g)
    c, ci = ess.color(ctx, other)
    assert torch.equal(c, plain) and ci["iterations"] == pi["iterations"], form
    jacobi, it = oracle.color_jacobi(off, col)
    assert np.array_equal(c.cpu().numpy(), jacobi) and ci["iterations"] == it, form
    other.close()


def _caller_buffers(n):
    """int32 `out` buffers a caller may hand over for n labels: (what, buffer)."""
    garbage = torch.randint(-2**31, 2**31 - 1, (n,), dtype=torch.int32, device="cuda")
    odd = _misaligned(torch.full((n,), SENTINEL, dtype=torch.int32, device="cuda"))
    longer = torch.full((n + 67,), SENTINEL, dtype=torch.int32, device="cuda")
    return [("garbage", garbage), ("misaligned", odd), ("longer than n", longer)]


def test_kcore_and_color_into_caller_buffers(ctx, multigraph, deep_peel):
    """`out` full of garbage, a misaligned view, a buffer longer than n (its tail untouched), one buffer reused across
    graphs; two runs byte-identical."""
    runs = {"kcore merge_path": lambda g, o: ess.kcore(ctx, g, lb="merge_path", out=o)[0],
            "kcore bucketing": lambda g, o: ess.kcore(ctx, g, lb="bucketing", out=o)[0],
            "color": lambda g, o: ess.color(ctx, g, out=o)[0]}
    for name, (_, g, _, _, _) in (("multigraph", multigraph), ("deep peel", deep_peel)):
        n = g.n
        for what, run in runs.items():
            plain = run(g, None)
            assert torch.equal(run(g, None), plain), (name, what, "two runs differ")
            for kind, buf in _caller_buffers(n):
                before = buf.clone()
                got = run(g, buf)
                assert got.data_ptr() == buf.data_ptr(), (name, what, kind)
                assert torch.equal(buf[:n], plain), (name, what, kind)
                assert torch.equal(buf[n:], before[n:]), (name, what, kind, "wrote past n")
    # one buffer handed to two graphs of different sizes in turn
    (_, g1, _, _, k1), (_, g2, _, _, k2) = multigraph, deep_peel
    big = max(g1.n, g2.n) + 32
    shared = torch.full((big,), SENTINEL, dtype=torch.int32, device="cuda")
    for g, want in ((g1, k1), (g2, k2), (g1, k1)):
        shared[g.n:] = SENTINEL
        ess.kcore(ctx, g, lb="block_mapped", out=shared)
        assert np.array_equal(shared[:g.n].cpu().numpy(), want)
        assert bool((shared[g.n:] == SENTINEL).all())
        c, _ = ess.color(ctx, g, out=shared)
        assert c.data_ptr() == shared.data_ptr()
        assert torch.equal(shared[:g.n], ess.color(ctx, g)[0])
        assert bool((shared[g.n:] == SENTINEL).all())


# ------------------------------------------------------------------------------------------------ colouring
@pytest.mark.parametrize("scale", [16, 18])
def test_color_rmat(ctx, s16, s18, scale):
    _, g, (off, col, _) = s16 if scale == 16 else s18
    c, info = ess.color(ctx, g)
    want, it = oracle.color_jacobi(off, col)
    got = c.cpu().numpy()
    assert np.array_equal(got, want), scale
    assert info["iterations"] == it
    assert oracle.color_errors(off, col, got) == 0


def _tie_graph(n, seed):
    """Every pair of vertices that draw the same random value in colouring's stream is joined by an edge; added to
    that: 4n random symmetric edges and a hub of 5000 neighbours. Returns (off, col, tied pairs)."""
    r = oracle.randoms(n, 0.0, float(n))
    order = np.argsort(r, kind="stable")
    rs = r[order]
    tu, tv = [], []
    j = 1
    while True:  # equal values are adjacent once sorted: pair every vertex with the next j-th one of equal value
        same = np.flatnonzero(rs[j:] == rs[:-j])
        if same.size == 0:
            break
        tu.append(order[same])
        tv.append(order[same + j])
        j += 1
    tu, tv = np.concatenate(tu), np.concatenate(tv)
    rng = np.random.default_rng(seed)
    u, v = rng.integers(0, n, 4 * n), rng.integers(0, n, 4 * n)
    keep = u != v
    hub = int(rng.integers(0, n))
    nbrs = rng.choice(np.delete(np.arange(n), hub), 5000, replace=False)
    off, col = _symmetric(n, np.concatenate([tu, u[keep], np.full(nbrs.size, hub)]),
                          np.concatenate([tv, v[keep], nbrs]))
    return off, col, tu.size


@pytest.mark.parametrize("scale", [16, 20])
def test_color_tie_break(ctx, scale):
    """Adjacent vertices with equal random values: the lower id cannot be the local maximum and the higher id cannot be
    the local minimum. Whichever of the two is coloured first, its colour depends on that rule, so each tied edge makes
    a flipped tie-break visible."""
    n = 1 << scale
    off, col, ties = _tie_graph(n, scale)
    assert ties >= 80, ties
    assert np.diff(off).max() >= BIG_DEGREE
    g = ess.Graph(_csr(off, col, "ties", True))
    c, info = ess.color(ctx, g)
    got = c.cpu().numpy()
    want, it = oracle.color_jacobi(off, col)
    assert np.array_equal(got, want), scale
    assert info["iterations"] == it
    assert oracle.color_errors(off, col, got) == 0


def test_color_multigraphs(ctx, multigraph):
    """Self-loops, parallel edges and isolated vertices: the Jacobi colours, and a valid colouring. On directed
    multigraphs only the Jacobi colours: a vertex does not see its in-neighbours, so validity is not promised."""
    _, g, off, col, _ = multigraph
    c, info = ess.color(ctx, g)
    want, it = oracle.color_jacobi(off, col)
    assert np.array_equal(c.cpu().numpy(), want) and info["iterations"] == it
    assert oracle.color_errors(off, col, want) == 0
    rng = np.random.default_rng(43)
    for trial in range(40):
        csr = _arbitrary_multigraph(rng)
        o, cl, _ = csr.host()
        c, info = ess.color(ctx, ess.Graph(csr))
        want, it = oracle.color_jacobi(o, cl)
        assert np.array_equal(c.cpu().numpy(), want), trial
        assert info["iterations"] == it, trial


# ------------------------------------------------------------------------------------------------ random stream
@pytest.mark.parametrize("lo,hi", [(0.0, None), (-3.5, 7.25), (1e6, 1e6 + 1)])
@pytest.mark.parametrize("n", [1 << 26, (1 << 20) + 37])
def test_random_stream(ctx, n, lo, hi):
    """generate::random::uniform_distribution: the oracle's stream bit for bit, past 2^26 elements and at a length that
    is not a multiple of the block size; (0, n) is the range colouring uses."""
    hi = float(n) if hi is None else hi
    got = ess.randoms(ctx, n, lo, hi).cpu().numpy()
    want = oracle.randoms(n, lo, hi)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (n, lo, hi)


# ------------------------------------------------------------------------------------------------ out= buffers
SOURCE = 3  # a vertex of rmat_s10 with 9 neighbours
ENTRY_POINTS = {
    "bfs": (torch.int32, lambda ctx, g, out: ess.bfs(ctx, g, SOURCE, out=out)),
    "sssp": (torch.float32, lambda ctx, g, out: ess.sssp(ctx, g, SOURCE, out=out)),
    "sssp_near_far": (torch.float32, lambda ctx, g, out: ess.sssp_near_far(ctx, g, SOURCE, out=out)),
    "sssp_delta": (torch.float32, lambda ctx, g, out: ess.sssp_delta(ctx, g, SOURCE, out=out)),
    "pagerank": (torch.float32, lambda ctx, g, out: ess.pagerank(ctx, g, out=out)),
    "ppr": (torch.float32, lambda ctx, g, out: ess.ppr(ctx, g, SOURCE, out=out)),
    "kcore": (torch.int32, lambda ctx, g, out: ess.kcore(ctx, g, out=out)),
    "color": (torch.int32, lambda ctx, g, out: ess.color(ctx, g, out=out)),
}


@pytest.fixture(scope="module")
def golden_graph(golden):
    """rmat_s10 (symmetric, weighted, 1024 vertices) from device arrays."""
    gd = golden["rmat_s10"]
    csr = gg.CSR(gd["offsets"].size - 1, gd["indices"].size, torch.from_numpy(gd["offsets"].astype(np.int32)).cuda(),
                 torch.from_numpy(gd["indices"]).cuda(), torch.from_numpy(gd["values"]).cuda(), "rmat_s10", True)
    return csr, ess.Graph(csr)


def _refused(ctx, run, g, out, what):
    launches = ctx.launches()
    with pytest.raises(ess.EssentialsError, match="CUDA tensor of at least"):
        run(ctx, g, out)
    assert ctx.launches() == launches, (what, "a kernel ran before the refusal")


@pytest.mark.parametrize("entry", list(ENTRY_POINTS))
def test_out_buffers_are_refused_before_any_launch(ctx, golden_graph, entry):
    """A wrong dtype, a host tensor, n - 1 elements and a strided view: each raises before a kernel runs."""
    dtype, run = ENTRY_POINTS[entry]
    _, g = golden_graph
    n = g.n
    bad = {
        "wrong dtype": torch.zeros(n, dtype=torch.float32 if dtype == torch.int32 else torch.int32, device="cuda"),
        "int64": torch.zeros(n, dtype=torch.int64, device="cuda"),
        "host tensor": torch.zeros(n, dtype=dtype),
        "n - 1 elements": torch.zeros(n - 1, dtype=dtype, device="cuda"),
        "strided view": torch.zeros(2 * n, dtype=dtype, device="cuda")[::2],
        "numpy array": np.zeros(n, np.int32 if dtype == torch.int32 else np.float32),
    }
    for what, out in bad.items():
        _refused(ctx, run, g, out, (entry, what))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs a second GPU")
@pytest.mark.parametrize("entry", list(ENTRY_POINTS))
def test_out_buffer_on_another_device_is_refused(ctx, golden_graph, entry):
    dtype, run = ENTRY_POINTS[entry]
    _, g = golden_graph
    _refused(ctx, run, g, torch.zeros(g.n, dtype=dtype, device="cuda:1"), (entry, "cuda:1"))


@pytest.mark.parametrize("entry", list(ENTRY_POINTS))
def test_out_buffers_misaligned_and_longer_are_accepted(ctx, golden_graph, entry):
    """A view 4 bytes past a 16-byte boundary that runs 37 elements past n: the result lands in its first n elements,
    the element before it and its tail stay untouched. Also a buffer allocated on plain "cuda" for a graph built from
    host arrays, as callers that time the host-array build do."""
    dtype, run = ENTRY_POINTS[entry]
    csr, g = golden_graph
    n = g.n
    plain, _ = run(ctx, g, None)
    buf = torch.full((n + 38,), SENTINEL, dtype=torch.int32, device="cuda").view(dtype)
    before = buf.clone()
    view = buf[1:]
    got, _ = run(ctx, g, view)
    assert got.data_ptr() == view.data_ptr() and view.data_ptr() % 16 == 4
    bits = lambda t: t.view(torch.int32)
    assert torch.equal(bits(buf[:1]), bits(before[:1])) and torch.equal(bits(buf[1 + n:]), bits(before[1 + n:])), entry
    if entry == "pagerank":  # dangling mass summed with float atomics: 1e-6 relative, the suite's bar
        assert torch.allclose(view[:n], plain, rtol=1e-6, atol=0), entry
    elif entry == "ppr":
        assert float((view[:n] - plain).abs().max()) <= 1e-6, entry
    else:
        assert torch.equal(bits(view[:n]), bits(plain)), entry
    gh = ess.Graph.from_host(ctx, csr.to("cpu"))
    assert gh.device == torch.empty(1, device="cuda").device
    out = torch.empty(n, dtype=dtype, device="cuda")
    got, _ = run(ctx, gh, out)
    assert got.data_ptr() == out.data_ptr()
    gh.close()
