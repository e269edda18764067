"""GPU suite (-m gpu): PageRank and personalised PageRank against float64 references written in this file.

The other PageRank tests run one directed RMAT with unit weights, whose largest in- and out-degrees stay below 1000.
The graphs here are built to reach every gather and scatter path of pr.hxx and of the advance it calls: in-degrees
on both sides of the pull bins (short_degree 8, hub_degree 4096) and one several CTA strides long, out-degrees of
4096 and ~6000 (the advance's grid-wide hub expansion, big_degree 4096), self-loops, duplicate edges, dangling and
isolated vertices, a vertex whose out-weights sum to 0, three weight variants and int64 offsets."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import essentials_b200 as ess
import oracle
from essentials_b200 import graphgen as gg

pytestmark = pytest.mark.gpu

LBS = list(ess.IMPLEMENTED_LOAD_BALANCERS)
ALPHA = float(np.float32(0.85))  # the kernels compute with the float alpha
KNOB_DEFAULTS = {"advance_engine": 1}
HUB_DEGREE = 4096  # b200::hub_degree (one CTA per row) and advance kernels::big_degree (grid-wide)
IN_HUB_DEGREES = (7, 8, 4095, 4096, 4097, 9001)
OUT_HUB_DEGREES = (4096, 6007)

# Tolerance of the pull path after 1-3 iterations. Per edge the kernel rounds to float a few times: iw = alpha/Σw,
# contrib = p·iw, contrib·w. It sums the terms of a row in double and rounds p to float once per iteration. That is
# at most about 4·2^-24 relative error per iteration, scaled by alpha <= 1, so 3 iterations stay below 2e-6.
# Dropping one edge of a 9000-edge row changes that row by about 1e-4, 50 times this bound; ignoring a weight in
# [1, 64) changes a row by far more.
PULL_RTOL = 2e-6


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


# ------------------------------------------------------------------------------------------------ references
def _matrix(off, col, w):
    """n x n scipy CSR; duplicate edges add up, which is what every sum over them does."""
    n = off.size - 1
    rows = np.repeat(np.arange(n), np.diff(off))
    data = np.ones(col.size) if w is None else w.astype(np.float64)
    return sp.csr_matrix((data, (rows, col.astype(np.int64))), shape=(n, n))


def pagerank_ref(off, col, w, iters, tol=0.0, alpha=ALPHA):
    """float64 restatement of the iteration in pr.hxx. Runs `iters` iterations, or stops after the first one whose
    max|p - plast| is below `tol`. Returns (p, iterations run)."""
    A = _matrix(off, col, w)
    n = A.shape[0]
    out_w = np.asarray(A.sum(axis=1)).ravel()
    iw = np.divide(alpha, out_w, out=np.zeros(n), where=out_w != 0)
    p = np.full(n, 1.0 / n)
    for k in range(1, iters + 1):
        plast = p
        dsum = alpha * plast[iw == 0].sum()
        p = (1 - alpha + dsum) / n + A.T @ (plast * iw)
        if np.abs(p - plast).max() < tol:
            break
    return p, k


def ppr_ref(off, col, seed, alpha=0.15, eps=1e-6):
    """float64 level-synchronous restatement of ppr.hxx. With positive updates a residual crosses its threshold at
    most once per level, whatever order the updates arrive in, so the next frontier is {v: before < th <= after}."""
    alpha, eps = float(np.float32(alpha)), float(np.float32(eps))
    A = _matrix(off, col, None)
    deg = np.diff(off).astype(np.float64)
    n = deg.size
    p, r = np.zeros(n), np.zeros(n)
    r[seed] = 1.0
    rp = r.copy()
    front = np.array([seed])
    while front.size:
        p[front] += 2 * alpha / (1 + alpha) * r[front]
        rp[front] = 0
        before = rp.copy()
        push = np.zeros(n)
        live = front[deg[front] > 0]
        push[live] = (1 - alpha) / (1 + alpha) * r[live] / deg[live]
        rp = rp + A.T @ push
        th = deg * eps
        front = np.flatnonzero((before < th) & (rp >= th))
        r = rp.copy()
    return p


# ------------------------------------------------------------------------------------------------ graphs
def multigraph_edges():
    """Directed multigraph on n = 30011 vertices (not a multiple of 32). Returns (n, src, dst, w, zero_out) with
    w = graphgen.pair_weights and zero weight on every out-edge of `zero_out`."""
    rng = np.random.default_rng(20261021)
    n = 30011
    ids = rng.permutation(n)
    in_hubs, out_hubs, zero_out = ids[:6], ids[6:8], ids[8]
    isolated, no_out, no_in, rest = ids[9:49], ids[49:649], ids[649:1249], ids[1249:]
    srcs = np.concatenate([rest, no_in, in_hubs])  # sources of the background edges
    dsts = np.concatenate([rest, no_out, out_hubs, [zero_out]])  # in-hubs get only their own edges
    m = 160000
    # skewed draws: in- and out-degrees from 0 up to ~1000, filling the warp bin [8, 4096)
    src = [srcs[(rng.random(m) ** 2 * srcs.size).astype(np.int64)]]
    dst = [dsts[(rng.random(m) ** 2 * dsts.size).astype(np.int64)]]
    loops = rng.choice(rest, 64, replace=False)
    src.append(loops), dst.append(loops)
    again = rng.integers(0, m, 2000)  # duplicate edges
    src.append(src[0][again]), dst.append(dst[0][again])
    for h, d in zip(in_hubs, IN_HUB_DEGREES):
        s = srcs[rng.integers(0, srcs.size, d)]
        if d == 9001:
            s[0] = h  # a self-loop on an in-hub
        if d == 4097:
            s[100:200] = s[:100]
        src.append(s), dst.append(np.full(d, h))
    for h, d in zip(out_hubs, OUT_HUB_DEGREES):
        t = dsts[rng.integers(0, dsts.size, d)]
        t[0] = h
        src.append(np.full(d, h)), dst.append(t)
    src.append(np.full(5, zero_out)), dst.append(dsts[rng.integers(0, dsts.size, 5)])
    src, dst = np.concatenate(src).astype(np.int64), np.concatenate(dst).astype(np.int64)
    w = gg.pair_weights(torch.from_numpy(src), torch.from_numpy(dst)).numpy()
    w[src == zero_out] = 0
    return n, src, dst, w, zero_out


def csr_arrays(n, src, dst, w=None):
    order = np.lexsort((dst, src))
    off = np.zeros(n + 1, np.int64)
    np.cumsum(np.bincount(src, minlength=n), out=off[1:])
    return off, dst[order], None if w is None else w[order]


def device_csr(off, col, w, name, symmetric=False, wide=False):
    return gg.CSR(off.size - 1, col.size, torch.from_numpy(off.astype(np.int64 if wide else np.int32)).cuda(),
                  torch.from_numpy(col.astype(np.int32)).cuda(),
                  None if w is None else torch.from_numpy(w.astype(np.float32)).cuda(), name, symmetric)


class Case:
    """A device graph, its host arrays and cached float64 references."""

    def __init__(self, csr, csc=None):
        self.csr, self.csc = csr, csc
        self.g = ess.Graph(csr, csc=csc)
        self.off, self.col, self.w = csr.host()
        self._refs = {}

    def ref(self, iters, tol=0.0, alpha=ALPHA):
        key = (iters, tol, alpha)
        if key not in self._refs:
            self._refs[key] = pagerank_ref(self.off, self.col, self.w, iters, tol, alpha)
        return self._refs[key]


GRAPHS = ["multi-none", "multi-ones", "multi-pair", "multi64-pair", "rmat16-hash"]


@pytest.fixture(scope="module")
def multi():
    n, src, dst, w, zero_out = multigraph_edges()
    off, col, w = csr_arrays(n, src, dst, w)
    out_deg, in_deg = np.diff(off), np.bincount(col, minlength=n)
    # the features the graph exists for
    for d in IN_HUB_DEGREES:
        assert np.count_nonzero(in_deg == d) >= 1, d
    assert np.count_nonzero(in_deg >= HUB_DEGREE) == 3 and in_deg.max() == 9001
    assert sorted(out_deg[out_deg >= HUB_DEGREE]) == list(OUT_HUB_DEGREES)
    loops = src[src == dst]
    assert loops.size > 64 and np.any(in_deg[loops] >= HUB_DEGREE) and np.any(out_deg[loops] >= HUB_DEGREE)
    assert np.unique(src * n + dst).size < src.size
    assert np.any((out_deg == 0) & (in_deg > 0)) and np.any((in_deg == 0) & (out_deg > 0))
    assert np.any((in_deg == 0) & (out_deg == 0))
    assert out_deg[zero_out] > 0 and not np.any(w[off[zero_out]:off[zero_out + 1]])
    assert n < 1 << 16 and n % 32 and np.count_nonzero((in_deg >= 8) & (in_deg < HUB_DEGREE)) > 1000
    return n, off, col, w


@pytest.fixture(scope="module")
def graphs(multi):
    n, off, col, w = multi
    out = {}
    for name, vals, wide in (("multi-none", None, False), ("multi-ones", np.ones_like(w), False),
                             ("multi-pair", w, False), ("multi64-pair", w, True)):
        csr = device_csr(off, col, vals, name, wide=wide)
        out[name] = Case(csr, ess.transpose(csr))
    rmat = gg.rmat_csr(16, weights="hash", device="cuda")  # symmetric: Graph(csr) gathers over the CSR itself
    deg = rmat.degrees().cpu().numpy()
    assert deg.max() >= 9000 and np.count_nonzero(deg >= HUB_DEGREE) >= 16
    out["rmat16-hash"] = Case(rmat)
    assert all(c.g.has_csc for c in out.values())
    return out


# ------------------------------------------------------------------------------------------------ (a) pull, 1-3 iterations
@pytest.mark.parametrize("iters", [1, 2, 3])
@pytest.mark.parametrize("name", GRAPHS)
def test_pull_matches_float64_after_few_iterations(ctx, graphs, name, iters):
    c = graphs[name]
    p, info = ess.pagerank(ctx, c.g, max_iterations=iters, pull=True)
    assert info["iterations"] == iters
    want, _ = c.ref(iters)
    got = p.cpu().numpy().astype(np.float64)
    rel = np.abs(got - want) / want
    assert rel.max() <= PULL_RTOL, (name, iters, rel.max(), int(rel.argmax()))


# ------------------------------------------------------------------------------------------------ (b) bit-exact push
def dyadic_graph():
    """Directed multigraph where one iteration at alpha 0.5 is exact in float in any summation order: n = 2^14, so
    p = 2^-14; every out-weight sum is a power of two, so iw = 0.5/Σw is one too; integer weights keep every term
    plast·iw·w and every rank a small multiple of a common power of two (checked by the test). Out-degrees 4096,
    4500 and 6000, an in-hub of ~6000, self-loops, duplicates, dangling vertices and a row of zero weights."""
    rng = np.random.default_rng(5)
    n = 1 << 14
    deg = rng.integers(0, 24, n)
    hubs = rng.choice(n, 4, replace=False)
    deg[hubs[:3]] = (4096, 4500, 6000)
    src = np.repeat(np.arange(n), deg)
    dst = rng.integers(0, n, src.size)
    dst[rng.random(src.size) < 0.03] = hubs[3]
    w = np.ones(src.size)
    start = np.concatenate([[0], np.cumsum(deg)])
    for v in np.flatnonzero(deg):
        s = 1 << int(deg[v] - 1).bit_length()  # the power of two >= deg
        w[start[v]:start[v + 1]] += rng.multinomial(s - deg[v], np.full(deg[v], 1.0 / deg[v]))
    zero = np.flatnonzero(deg == 5)[0]
    w[start[zero]:start[zero + 1]] = 0
    return n, src, dst, w


@pytest.fixture(scope="module")
def dyadic():
    n, src, dst, w = dyadic_graph()
    off, col, w = csr_arrays(n, src, dst, w)
    csr = device_csr(off, col, w, "dyadic")
    c = Case(csr, ess.transpose(csr))
    assert np.diff(c.off).max() >= 6000 and np.bincount(col, minlength=n).max() >= HUB_DEGREE
    return c


def test_pull_and_every_push_balancer_bit_exact_on_dyadic_graph(ctx, dyadic):
    c = dyadic
    alpha = 0.5
    want, _ = c.ref(1, alpha=alpha)
    # precondition: every term (the teleport base and each plast·iw·w) and every rank is an integer multiple of
    # one power of two 2^-k, and every rank is below 2^24 of them. Partial sums of such terms, in any order, are
    # integers below 2^24 in that unit, which float holds exactly.
    n = c.off.size - 1
    out_w = np.asarray(_matrix(c.off, c.col, c.w).sum(axis=1)).ravel()
    iw = np.divide(alpha, out_w, out=np.zeros(n), where=out_w != 0)
    src = np.repeat(np.arange(n), np.diff(c.off))
    terms = np.concatenate([[(1 - alpha + alpha * (iw == 0).sum() / n) / n], iw[src] * c.w / n])
    k = next(k for k in range(80) if np.all(np.mod(np.ldexp(terms, k), 1) == 0))
    units = np.ldexp(want, k)
    assert np.all(np.mod(units, 1) == 0) and units.max() < 2**24, (k, units.max())
    runs = [("pull", None)] + [(lb, engine) for lb in LBS for engine in (1, 0)]
    for lb, engine in runs:
        if engine is None:
            p, info = ess.pagerank(ctx, c.g, alpha=alpha, max_iterations=1, pull=True)
        else:
            with knob("advance_engine", engine):
                p, info = ess.pagerank(ctx, c.g, alpha=alpha, max_iterations=1, lb=lb, pull=False)
        got = p.cpu().numpy().astype(np.float64)
        assert info["iterations"] == 1
        assert np.array_equal(got, want), (lb, engine, np.count_nonzero(got != want), int(np.argmax(got != want)))


# ------------------------------------------------------------------------------------------------ (c) to convergence
@pytest.mark.parametrize("mode", ["pull"] + LBS)
@pytest.mark.parametrize("name", GRAPHS)
def test_converged_ranks_match_float64(ctx, graphs, name, mode):
    c = graphs[name]
    pull = mode == "pull"
    p, info = ess.pagerank(ctx, c.g, lb="block_mapped" if pull else mode, pull=pull)
    _, k_ref = c.ref(1000, tol=float(np.float32(1e-6)))
    assert abs(info["iterations"] - k_ref) <= 1, (info["iterations"], k_ref)
    want, _ = c.ref(info["iterations"])
    got = p.cpu().numpy().astype(np.float64)
    assert abs(got.sum() - 1.0) < 1e-5, got.sum()
    rel = np.abs(got - want) / want
    if pull:
        assert rel.max() <= 1e-6, (name, rel.max(), int(rel.argmax()))
    else:  # float atomics sum in whatever order the hardware schedules them
        assert rel.max() <= 1e-4, (name, mode, rel.max(), int(rel.argmax()))
        assert np.abs(got - want).sum() / want.sum() <= 1e-6, (name, mode)


# ------------------------------------------------------------------------------------------------ (d) edge cases
def _tiny(n, src, dst):
    off, col, _ = csr_arrays(n, np.asarray(src, np.int64), np.asarray(dst, np.int64))
    csr = device_csr(off, col, None, f"tiny-{n}")
    return Case(csr, device_csr(*csr_arrays(n, np.asarray(dst, np.int64), np.asarray(src, np.int64)), "tiny-T"))


@pytest.mark.parametrize("mode", ["pull"] + LBS)
def test_tiny_graphs(ctx, mode):
    pull = mode == "pull"
    run = lambda c: ess.pagerank(ctx, c.g, lb="block_mapped" if pull else mode, pull=pull)
    for n in (1, 37):  # no edges: all mass is dangling, so every rank stays 1/n
        p, info = run(_tiny(n, [], []))
        assert info["iterations"] == 1
        assert np.array_equal(p.cpu().numpy(), np.full(n, np.float32(1.0 / n))), (n, p)
    c = _tiny(1, [0], [0])  # one vertex with a self-loop
    p, info = run(c)
    assert info["iterations"] == 1 and abs(float(p[0]) - 1.0) <= 2e-7, p


def test_max_iterations_1_on_the_default_paths(ctx, graphs):
    for name in ("multi-pair", "rmat16-hash"):
        c = graphs[name]
        p, info = ess.pagerank(ctx, c.g, max_iterations=1)  # gathers: both graphs have an in-edge view
        assert info["iterations"] == 1
        assert np.allclose(p.cpu().numpy(), c.ref(1)[0], rtol=PULL_RTOL, atol=0), name
    c = graphs["multi-pair"]
    p, info = ess.pagerank(ctx, ess.Graph(c.csr), max_iterations=1)  # no CSC: scatters
    assert info["iterations"] == 1
    assert np.allclose(p.cpu().numpy(), c.ref(1)[0], rtol=1e-4, atol=0)


# ------------------------------------------------------------------------------------------------ (e) weights on one view
def test_pull_refuses_weights_on_only_one_view(ctx, graphs):
    """The gather multiplies by the CSC weights and iweights divides by the CSR weight sums: weights on only one of
    the two views would give wrong ranks without a word, so the pull path refuses the graph."""
    c = graphs["multi-pair"]
    bare = lambda v: gg.CSR(v.n, v.m, v.offsets, v.indices, None, v.name, v.symmetric)
    for csr, csc in ((c.csr, bare(c.csc)), (bare(c.csr), c.csc)):
        g = ess.Graph(csr, csc=csc)
        for pull in (True, None):
            with pytest.raises(ess.EssentialsError, match="weights"):
                ess.pagerank(ctx, g, max_iterations=2, pull=pull)
    g = ess.Graph(c.csr, csc=bare(c.csc))  # the scatter reads only the CSR: still the weighted answer
    p, _ = ess.pagerank(ctx, g, max_iterations=2, pull=False)
    assert np.allclose(p.cpu().numpy(), c.ref(2)[0], rtol=1e-4, atol=0)


# ------------------------------------------------------------------------------------------------ PPR
@pytest.fixture(scope="module")
def ppr_graphs(multi):
    n, off, col, _ = multi
    src = np.repeat(np.arange(n), np.diff(off))
    loop = src == col
    sym = csr_arrays(n, np.concatenate([src, col[~loop]]), np.concatenate([col, src[~loop]]))
    out = {"multi-sym": (ess.Graph(device_csr(sym[0], sym[1], None, "multi-sym", symmetric=True)), sym[0], sym[1])}
    rmat = gg.rmat_csr(16, device="cuda")
    out["rmat16"] = (ess.Graph(rmat),) + rmat.host()[:2]
    seeds = {}
    for name, (_, off, _) in out.items():
        deg = np.diff(off)
        assert deg.max() >= HUB_DEGREE
        seeds[name] = {"hub": int(deg.argmax()), "degree-1": int(np.flatnonzero(deg == 1)[0]),
                       "isolated": int(np.flatnonzero(deg == 0)[0])}
    return out, seeds


@pytest.mark.parametrize("lb", LBS)
@pytest.mark.parametrize("name", ["multi-sym", "rmat16"])
def test_ppr_matches_oracle_and_float64(ctx, ppr_graphs, name, lb):
    (g, off, col), seeds = ppr_graphs[0][name], ppr_graphs[1][name]
    a = np.float32(0.15)
    for kind, s in seeds.items():
        got = ess.ppr(ctx, g, s, lb=lb)[0].cpu().numpy()
        if kind == "isolated":
            want = np.zeros_like(got)
            want[s] = np.float32(2 * a) / np.float32(1 + a)
            assert np.array_equal(got, want), (name, lb, s)
            continue
        err = np.abs(got - oracle.ppr(off, col, s)).max()
        assert err <= 1e-6, (name, lb, kind, err)
        want = ppr_ref(off, col, s)
        got = got.astype(np.float64)
        assert np.abs(got - want).sum() / want.sum() <= 1e-5, (name, lb, kind)
        assert got.min() >= 0 and got.sum() <= 1 + 1e-6, (name, lb, kind, got.sum())
