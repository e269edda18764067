"""GPU suite (-m gpu): the CUDA path, called through the C ABI, against the oracle and the golden vectors.

Bars: BFS depths, k-core numbers, colours, operator outputs — bit-exact. SSSP — bit-exact (stronger than the
1e-6 relative north_star asks). PageRank — 1e-6 relative per element on the default (gather) path; the
reference-style scatter (pull=False: unordered float atomics, like the reference) — 1e-6 relative in L1 and
1e-4 per element. PPR — 1e-6 absolute, the reference driver's own tolerance
(examples/algorithms/ppr/ppr.cu:76-79)."""
import numpy as np
import pytest
import torch

import essentials_b200 as ess
import oracle
from essentials_b200 import graphgen as gg

pytestmark = pytest.mark.gpu

LBS = list(ess.IMPLEMENTED_LOAD_BALANCERS)
INF = 2**31 - 1


@pytest.fixture(scope="module")
def ctx():
    assert torch.cuda.is_available(), "GPU suite needs a CUDA device"
    return ess.Context(0)


def csr_from_golden(g, wide=False):
    off = torch.from_numpy(g["offsets"].astype(np.int64 if wide else np.int32)).cuda()
    return gg.CSR(off.numel() - 1, g["indices"].size, off, torch.from_numpy(g["indices"]).cuda(),
                  torch.from_numpy(g["values"]).cuda(), "golden", True)


@pytest.fixture(scope="module")
def graphs(golden):
    return {k: ess.Graph(csr_from_golden(v)) for k, v in golden.items()}


@pytest.fixture(scope="module")
def s16():
    csr = gg.rmat_csr(16, device="cuda")
    return csr, ess.Graph(csr), csr.host()


# ------------------------------------------------------------------------------------------------ BFS
@pytest.mark.parametrize("direction", ["forward", "optimized"])
@pytest.mark.parametrize("lb", LBS)
@pytest.mark.parametrize("name", ["chesapeake", "rmat_s10", "grid_24x17"])
def test_bfs_golden(ctx, graphs, golden, name, lb, direction):
    for s in golden[name]["sources"]:
        depth, info = ess.bfs(ctx, graphs[name], int(s), lb=lb, direction=direction)
        assert np.array_equal(depth.cpu().numpy(), golden[name][f"bfs_{s}"]), (name, lb, direction, int(s))
        assert info["iterations"] >= 1


@pytest.mark.parametrize("direction", ["forward", "optimized"])
@pytest.mark.parametrize("lb", LBS)
def test_bfs_config1_rmat_scale16(ctx, s16, lb, direction):
    """BASELINE config 1: RMAT scale-16 ef-16 vs the CPU reference; source 0 (what the reference driver
    hard-codes, bfs.cu:62) and seeded non-isolated sources."""
    csr, g, (off, col, _) = s16
    for s in [0] + gg.pick_sources(csr, 3):
        depth, info = ess.bfs(ctx, g, s, lb=lb, direction=direction)
        assert np.array_equal(depth.cpu().numpy(), oracle.bfs(off, col, s)), (lb, direction, s)
    if direction == "optimized":
        assert info["pull_steps"] >= 1, "a Kronecker graph must trigger the bottom-up switch"


def test_bfs_int64_offsets(ctx, golden):
    g = ess.Graph(csr_from_golden(golden["rmat_s10"], wide=True))
    for lb in LBS:
        for direction in ("forward", "optimized"):
            s = int(golden["rmat_s10"]["sources"][0])
            depth, _ = ess.bfs(ctx, g, s, lb=lb, direction=direction)
            assert np.array_equal(depth.cpu().numpy(), golden["rmat_s10"][f"bfs_{s}"])


@pytest.mark.parametrize("wide", [False, True])
def test_graph_from_host_arrays(ctx, s16, wide):
    """ess_graph_create_from_host (the reference drivers' host csr_t -> device vectors -> from_csr,
    examples/algorithms/bfs/bfs.cu:25-66): chunked H2D on a copy stream with the bottom-up hints built per arrived
    chunk. Chunks of 4096 edges make the scale-16 graph cross ~500 chunk boundaries (vertices whose lists straddle a
    boundary, hubs that span several chunks); depths and distances must equal the device-array graph, pinned or
    pageable host memory, 32- or 64-bit offsets, and the counters must show the hinted bottom-up levels."""
    csr, g, (off, col, _) = s16
    src = gg.pick_sources(csr, 2)
    ess.tune("host_chunk_edges", 4096)
    try:
        for pinned in (True, False):
            host = csr.pinned() if pinned else csr.to("cpu")
            if wide:
                host = gg.CSR(host.n, host.m, host.offsets.long(), host.indices, host.values, host.name, host.symmetric)
                if pinned:
                    host = host.pinned()
            gh = ess.Graph.from_host(ctx, host)
            assert gh.has_csc and gh.offset_bits == (64 if wide else 32)
            for s in src:
                for lb, direction in (("merge_path", "optimized"), ("block_mapped", "forward")):
                    want, i0 = ess.bfs(ctx, g, s, lb=lb, direction=direction)
                    got, i1 = ess.bfs(ctx, gh, s, lb=lb, direction=direction)
                    assert torch.equal(want, got), (pinned, wide, s, lb, direction)
                    assert np.array_equal(got.cpu().numpy(), oracle.bfs(off, col, s))
                    if direction == "optimized" and not wide:
                        assert i1["pull_steps"] == i0["pull_steps"] >= 1
                        for k in ("pull_vertices", "pull_misses", "pull_found"):  # same hints -> same bottom-up work
                            assert i1[k] == i0[k], (k, i0, i1)
            gh.close()
        weighted = gg.rmat_csr(12, weights="hash", device="cpu")  # the values array travels last
        gw, gd = ess.Graph.from_host(ctx, weighted.pinned()), ess.Graph(weighted.to("cuda"))
        for s in gg.pick_sources(weighted, 2):
            assert torch.equal(ess.sssp(ctx, gw, s)[0], ess.sssp(ctx, gd, s)[0])
        gw.close()
    finally:
        ess.tune("host_chunk_edges", 64 << 20)
    with pytest.raises(ess.EssentialsError):
        ess.Graph.from_host(ctx, csr)  # device tensors belong to Graph(csr)
    bad = csr.to("cpu")
    bad = gg.CSR(bad.n, bad.m, bad.offsets.clone(), bad.indices, None, "", True)
    bad.offsets[-1] += 1
    with pytest.raises(ess.EssentialsError, match="row_offsets"):
        ess.Graph.from_host(ctx, bad)
    directed = ess.Graph.from_host(ctx, gg.rmat_csr(8, symmetric=False, device="cpu"), symmetric=False)
    assert not directed.has_csc
    d, _ = ess.bfs(ctx, directed, 0)
    assert int(d[0]) == 0
    with pytest.raises(ess.EssentialsError):
        ess.bfs(ctx, directed, 0, direction="optimized")


def test_bfs_isolated_source_and_errors(ctx, s16):
    csr, g, (off, col, _) = s16
    iso = int(torch.nonzero(csr.degrees() == 0)[0])
    for direction in ("forward", "optimized"):
        depth, info = ess.bfs(ctx, g, iso, direction=direction)
        d = depth.cpu().numpy()
        assert d[iso] == 0 and (d != INF).sum() == 1
    with pytest.raises(ess.EssentialsError):
        ess.bfs(ctx, g, csr.n)  # source out of range
    with pytest.raises(ess.EssentialsError):
        ess.bfs(ctx, g, 0, lb="warp_mapped")  # "Advance type not supported." like the reference
    directed = ess.Graph(gg.rmat_csr(8, symmetric=False, device="cuda"))
    with pytest.raises(ess.EssentialsError):
        ess.bfs(ctx, directed, 0, direction="optimized")  # needs CSR and CSC


def test_bfs_large_properties(ctx):
    """Size-independent checks at a scale the CPU oracle is not needed for (scale-20): all variants agree,
    every edge spans at most one level, every reached non-source vertex has a parent one level up."""
    csr = gg.rmat_csr(20, device="cuda")
    g = ess.Graph(csr)
    s = gg.pick_sources(csr, 1)[0]
    base, _ = ess.bfs(ctx, g, s, lb="block_mapped", direction="forward")
    for lb in LBS:
        d2, info = ess.bfs(ctx, g, s, lb=lb, direction="optimized")
        assert torch.equal(base, d2), lb
    rows = torch.repeat_interleave(torch.arange(csr.n, device="cuda"), csr.degrees().long())
    du, dv = base[rows].long(), base[csr.indices.long()].long()
    assert bool(((du == INF) == (dv == INF)).all()), "reached set is closed under edges"
    ok = du != INF
    assert int((du[ok] - dv[ok]).abs().max()) <= 1
    has_parent = torch.zeros(csr.n, dtype=torch.bool, device="cuda")
    has_parent[rows[ok & (dv == du - 1)]] = True
    reached = base != INF
    reached[s] = False
    assert bool(has_parent[reached].all())


# ------------------------------------------------------------------------------------------------ SSSP
@pytest.mark.parametrize("lb", LBS)
@pytest.mark.parametrize("name", ["chesapeake", "rmat_s10", "grid_24x17"])
def test_sssp_golden_bit_exact(ctx, graphs, golden, name, lb):
    for s in golden[name]["sources"]:
        dist, _ = ess.sssp(ctx, graphs[name], int(s), lb=lb)
        assert np.array_equal(dist.cpu().numpy(), golden[name][f"sssp_{s}"]), (name, lb, int(s))


@pytest.mark.parametrize("lb", ["block_mapped", "merge_path", "bucketing"])
def test_sssp_rmat14_and_grid(ctx, lb):
    csr = gg.rmat_csr(14, weights="hash", device="cuda")
    off, col, val = csr.host()
    g = ess.Graph(csr)
    for s in gg.pick_sources(csr, 2):
        dist, _ = ess.sssp(ctx, g, s, lb=lb)
        want = oracle.sssp(off, col, val, s)
        got = dist.cpu().numpy()
        assert np.array_equal(got, want), f"max rel err {np.max(np.abs(got - want) / np.maximum(want, 1e-30))}"
    grid = gg.grid_csr(96, 80, device="cuda")
    off, col, val = grid.host()
    dist, info = ess.sssp(ctx, ess.Graph(grid), 0, lb=lb)
    assert np.array_equal(dist.cpu().numpy(), oracle.sssp(off, col, val, 0))
    assert info["iterations"] >= 96 + 80 - 2


@pytest.mark.parametrize("delta", [0.0, 1.0, 7.5, 64.0, 1e9])
def test_sssp_near_far_bit_exact(ctx, graphs, golden, delta):
    """operators::advance::execute_near_far (persistent near/far kernel) must give the reference distances for
    every bucket width: delta -> inf degenerates to plain label correcting, tiny delta to Dijkstra order."""
    for name in ("chesapeake", "rmat_s10", "grid_24x17"):
        for s in golden[name]["sources"]:
            dist, info = ess.sssp_near_far(ctx, graphs[name], int(s), delta=delta)
            assert np.array_equal(dist.cpu().numpy(), golden[name][f"sssp_{s}"]), (name, int(s), delta)
            assert info["levels"] >= 1


def test_sssp_near_far_larger_graphs(ctx):
    csr = gg.rmat_csr(14, weights="hash", device="cuda")  # hubs: exercises the warp-cooperative walk
    off, col, val = csr.host()
    g = ess.Graph(csr)
    for s in gg.pick_sources(csr, 2):
        dist, info = ess.sssp_near_far(ctx, g, s)
        assert np.array_equal(dist.cpu().numpy(), oracle.sssp(off, col, val, s))
    grid = gg.grid_csr(300, 200, device="cuda")
    off, col, val = grid.host()
    want = oracle.sssp(off, col, val, 17)
    for delta in (0.0, 16.0, 200.0):
        dist, info = ess.sssp_near_far(ctx, ess.Graph(grid), 17, delta=delta)
        assert np.array_equal(dist.cpu().numpy(), want), delta
        assert info["relaxations"] >= grid.m * 0 + 1


def test_sssp_near_far_long_runs(ctx):
    """One launch of the persistent near-far kernel over hundreds of small levels (a long, thin grid) and over the wide
    levels of a Kronecker graph: distances bit-equal to the oracle."""
    grid = gg.grid_csr(211, 97, device="cuda")
    off, col, val = grid.host()
    dist, info = ess.sssp_near_far(ctx, ess.Graph(grid), 5)
    assert np.array_equal(dist.cpu().numpy(), oracle.sssp(off, col, val, 5))
    assert info["levels"] > 200
    csr = gg.rmat_csr(17, weights="hash", device="cuda")
    off, col, val = csr.host()
    s = gg.pick_sources(csr, 1)[0]
    dist, info = ess.sssp_near_far(ctx, ess.Graph(csr), s)
    assert np.array_equal(dist.cpu().numpy(), oracle.sssp(off, col, val, s))


def test_sssp_thresholds_make_progress_on_extreme_weight_ranges(ctx):
    """Weights {1e-3, 1e6}: distances reach ~1e7 while delta stays ~1e-3, so (floor(d / delta) + 1) * delta and
    threshold + delta both round to <= d in float; the near-far kernel and run_delta must still advance (they step
    to nextafter(d)) instead of spinning, and the distances stay bit-exact."""
    import dataclasses
    grid = gg.grid_csr(40, 30, device="cuda")
    rows = torch.repeat_interleave(torch.arange(grid.n, device="cuda"), grid.degrees().long())
    lo, hi = torch.minimum(rows, grid.indices.long()), torch.maximum(rows, grid.indices.long())
    w = torch.where(((lo * 31 + hi) % 5) == 0, 1e6, 1e-3).to(torch.float32)  # symmetric: both directions agree
    g2 = dataclasses.replace(grid, values=w)
    off, col, val = g2.host()
    want = oracle.sssp(off, col, val, 0)
    g = ess.Graph(g2)
    d_nf, _ = ess.sssp_near_far(ctx, g, 0, delta=1e-3)
    assert np.array_equal(d_nf.cpu().numpy(), want)
    d_dl, _ = ess.sssp_delta(ctx, g, 0, delta=1e-3)
    assert np.array_equal(d_dl.cpu().numpy(), want)


def test_atomic_wrappers_return_the_old_value(ctx):
    """math::atomic::{add,min,max,exch} hand back what the cell held BEFORE the update (user lambdas compare against
    it: bfs `iteration + 1 < old`, sssp `candidate < old`); float min/max are single ordered-integer atomics here
    (CAS loops in the reference), so negative values, zeros of both signs and infinities are checked explicitly."""
    vals = torch.tensor([5.5, -2.25, 7.0, -2.25, float("inf"), -0.0, 0.0, -1e30, 3.0, float("-inf"), 1.0],
                        dtype=torch.float32, device="cuda")
    for op, fold in (("min", np.minimum), ("max", np.maximum), ("add", np.add), ("exch", lambda a, b: b)):
        cell = torch.tensor([4.0], dtype=torch.float32, device="cuda")
        v = vals if op != "add" else torch.tensor([0.5, -2.25, 7.0, 1.0, 3.0], dtype=torch.float32, device="cuda")
        old = ess.atomic_probe(ctx, op, cell, v, serial=True).cpu().numpy()
        run = np.float32(4.0)
        for i, x in enumerate(v.cpu().numpy()):
            assert old[i] == run and np.signbit(old[i]) == np.signbit(run), (op, i, old[i], run)
            run = np.float32(fold(run, x))
        assert cell.item() == run
    ints = torch.tensor([9, -3, 12, -3, 2**31 - 1, -2**31, 0], dtype=torch.int32, device="cuda")
    for op, fold in (("min", min), ("max", max), ("exch", lambda a, b: b)):
        cell = torch.tensor([4], dtype=torch.int32, device="cuda")
        old = ess.atomic_probe(ctx, op, cell, ints, serial=True).cpu().numpy()
        run = 4
        for i, x in enumerate(ints.cpu().tolist()):
            assert int(old[i]) == run, (op, i)
            run = fold(run, x)
        assert cell.item() == run
    # concurrent: the returned values are exactly the successive contents of the cell
    big = (torch.rand(1 << 16, device="cuda") * 2000 - 1000).to(torch.float32)
    cell = torch.tensor([2000.0], dtype=torch.float32, device="cuda")
    old = ess.atomic_probe(ctx, "min", cell, big).cpu().numpy()
    assert cell.item() == big.min().item()
    improved = old > big.cpu().numpy()  # calls that lowered the cell: their `old` values are all distinct cell states
    states = np.sort(old[improved])[::-1]
    assert states[0] == 2000.0 and np.all(np.diff(states) < 0)
    assert np.all(old >= cell.item())
    total = torch.tensor([0], dtype=torch.int32, device="cuda")
    ones = torch.ones(1 << 16, dtype=torch.int32, device="cuda")
    old = ess.atomic_probe(ctx, "add", total, ones).cpu().numpy()
    assert total.item() == 1 << 16 and np.array_equal(np.sort(old), np.arange(1 << 16))


@pytest.mark.parametrize("fused", [0, 1])
@pytest.mark.parametrize("lb", LBS)
def test_sssp_fused_unique_level_loop(ctx, graphs, golden, lb, fused):
    """gunrock::sssp with operators::advance::execute_unique (default) and with the reference's advance + bypass
    filter pair (knob 0): same distances."""
    ess.tune("sssp_fused_unique", fused)
    try:
        for name in ("chesapeake", "rmat_s10", "grid_24x17"):
            for s in golden[name]["sources"]:
                dist, info = ess.sssp(ctx, graphs[name], int(s), lb=lb)
                assert np.array_equal(dist.cpu().numpy(), golden[name][f"sssp_{s}"]), (name, int(s), lb)
    finally:
        ess.tune("sssp_fused_unique", 1)


@pytest.mark.parametrize("delta", [0.0, 0.5, 7.5, 64.0, 3e38])
def test_sssp_delta_bit_exact(ctx, graphs, golden, delta):
    """gunrock::sssp::run_delta (dense active set, threshold advancing by delta): reference distances for every
    bucket width — huge delta is plain label correcting, tiny delta close to Dijkstra order — and n not a
    multiple of the 4-wide vector loads (chesapeake: 39 vertices)."""
    for name in ("chesapeake", "rmat_s10", "grid_24x17"):
        for s in golden[name]["sources"]:
            dist, info = ess.sssp_delta(ctx, graphs[name], int(s), delta=delta)
            assert np.array_equal(dist.cpu().numpy(), golden[name][f"sssp_{s}"]), (name, int(s), delta)
            assert info["passes"] >= info["rounds"] + 1  # the last pass finds nothing left


def test_sssp_delta_larger_graph_and_work(ctx):
    csr = gg.rmat_csr(15, weights="hash", device="cuda")
    off, col, val = csr.host()
    g = ess.Graph(csr)
    for s in gg.pick_sources(csr, 2):
        want = oracle.sssp(off, col, val, s)
        plain, i_plain = ess.sssp_delta(ctx, g, s, delta=3e38)
        near, i_near = ess.sssp_delta(ctx, g, s)
        assert np.array_equal(plain.cpu().numpy(), want) and np.array_equal(near.cpu().numpy(), want)
        # thresholds trade rounds for work: more rounds, fewer vertex expansions than plain label correcting
        assert i_near["rounds"] >= i_plain["rounds"] and i_near["expanded_vertices"] <= i_plain["expanded_vertices"]
    iso = int(torch.nonzero(csr.degrees() == 0)[0])
    dist, info = ess.sssp_delta(ctx, g, iso)
    d = dist.cpu().numpy()
    assert d[iso] == 0 and (np.delete(d, iso) == np.float32(3.4028234663852886e38)).all() and info["rounds"] == 1


def _arbitrary_multigraph(rng):
    """Small directed multigraph with self loops, parallel edges, isolated vertices, zero and tied weights."""
    n = int(rng.integers(2, 70))
    m = int(rng.integers(1, 400))
    src, dst = rng.integers(0, n, m), rng.integers(0, n, m)
    w = rng.choice(np.array([0.0, 0.5, 1.0, 1.0, 2.25, 7.0, 63.984375], np.float32), m)
    order = np.lexsort((dst, src))
    off = np.zeros(n + 1, np.int64)
    np.add.at(off, src + 1, 1)
    off = np.cumsum(off).astype(np.int32)
    return gg.CSR(n, m, torch.from_numpy(off).cuda(), torch.from_numpy(dst[order].astype(np.int32)).cuda(),
                  torch.from_numpy(w[order]).cuda(), "arbitrary", False)


def test_traversals_on_arbitrary_directed_multigraphs(ctx):
    """The degenerate inputs the oracle property test feeds the reference's CPU code, through every CUDA traversal:
    forward BFS with each balancer, push/pull BFS over CSR + transposed CSC, SSSP as frontier recipe (fused and
    reference pair), dense delta and near-far — all bit-equal to the oracle."""
    rng = np.random.default_rng(77)
    for trial in range(40):
        csr = _arbitrary_multigraph(rng)
        off, col, val = csr.host()
        g = ess.Graph(csr, csc=ess.transpose(csr))
        for s in {0, int(rng.integers(0, csr.n))}:
            want_bfs, want_sssp = oracle.bfs(off, col, s), oracle.sssp(off, col, val, s)
            for lb in LBS:
                d, _ = ess.bfs(ctx, g, s, lb=lb)
                assert np.array_equal(d.cpu().numpy(), want_bfs), (trial, s, lb)
            d, _ = ess.bfs(ctx, g, s, lb="merge_path", direction="optimized")
            assert np.array_equal(d.cpu().numpy(), want_bfs), (trial, s, "optimized")
            for fused in (1, 0):
                ess.tune("sssp_fused_unique", fused)
                d, _ = ess.sssp(ctx, g, s, lb="merge_path")
                assert np.array_equal(d.cpu().numpy(), want_sssp), (trial, s, "frontier", fused)
            ess.tune("sssp_fused_unique", 1)
            for delta in (0.0, 1.0, 3e38):
                d, _ = ess.sssp_delta(ctx, g, s, delta=delta)
                assert np.array_equal(d.cpu().numpy(), want_sssp), (trial, s, "delta", delta)
            d, _ = ess.sssp_near_far(ctx, g, s, delta=1.5)
            assert np.array_equal(d.cpu().numpy(), want_sssp), (trial, s, "near_far")


# ------------------------------------------------------------------------------------------------ PageRank
@pytest.mark.parametrize("mode", ["default", "pull", "block_mapped", "merge_path", "bucketing", "thread_mapped"])
def test_pagerank_directed_rmat(ctx, mode):
    """BASELINE config 4 shape at scale-12: directed RMAT, weights 1, alpha .85, tol 1e-6 (pr.cu:55-56)."""
    csr = gg.rmat_csr(12, symmetric=False, weights="ones", device="cuda")
    off, col, val = csr.host()
    csc = ess.transpose(csr)
    g = ess.Graph(csr, csc=csc)
    pull = mode in ("pull", "default")  # the default call gathers when the graph has an in-edge view: the 1e-6 path
    if mode == "default":
        p, info = ess.pagerank(ctx, g)
    else:
        p, info = ess.pagerank(ctx, g, lb="block_mapped" if pull else mode, pull=pull)
    got = p.cpu().numpy().astype(np.float64)
    _, it_cpu = oracle.pagerank(off, col, val)
    assert abs(info["iterations"] - it_cpu) <= 1, (info, it_cpu)
    want = oracle.pagerank(off, col, val, force_iters=info["iterations"])[0].astype(np.float64)
    assert abs(got.sum() - 1.0) < 1e-4
    rel_l1 = np.abs(got - want).sum() / want.sum()
    assert rel_l1 < 1e-6, rel_l1
    rtol = 1e-6 if pull else 1e-4  # push sums with unordered float atomics, exactly like the reference
    assert np.allclose(got, want, rtol=rtol, atol=0), np.max(np.abs(got - want) / want)


# ------------------------------------------------------------------------------------------------ PPR
@pytest.mark.parametrize("lb", LBS)
def test_ppr_golden(ctx, graphs, golden, lb):
    for name in ("chesapeake", "rmat_s10"):
        for s in golden[name]["ppr_seeds"]:
            p, _ = ess.ppr(ctx, graphs[name], int(s), lb=lb)
            err = np.abs(p.cpu().numpy() - golden[name][f"ppr_{s}"]).max()
            assert err <= 1e-6, (name, lb, int(s), err)


# ------------------------------------------------------------------------------------------------ k-core / colouring
@pytest.mark.parametrize("lb", LBS)
def test_kcore_golden(ctx, graphs, golden, lb):
    for name in ("chesapeake", "rmat_s10", "grid_24x17"):
        k, _ = ess.kcore(ctx, graphs[name], lb=lb)
        assert np.array_equal(k.cpu().numpy(), golden[name]["kcore"]), (name, lb)


def test_kcore_rmat12(ctx):
    csr = gg.rmat_csr(12, device="cuda")
    off, col, _ = csr.host()
    k, _ = ess.kcore(ctx, ess.Graph(csr), lb="merge_path")
    assert np.array_equal(k.cpu().numpy(), oracle.kcore(off, col))


def test_randoms_and_color(ctx, graphs, golden, s16):
    for name in ("chesapeake", "rmat_s10", "grid_24x17"):
        n = golden[name]["offsets"].size - 1
        r = ess.randoms(ctx, n, 0.0, float(n))
        assert np.array_equal(r.cpu().numpy(), golden[name]["randoms"]), "minstd stream differs from the reference's"
        c, info = ess.color(ctx, graphs[name])
        want, it = oracle.color_jacobi(golden[name]["offsets"], golden[name]["indices"], golden[name]["randoms"])
        assert np.array_equal(c.cpu().numpy(), want), name
        assert info["iterations"] == it
        assert oracle.color_errors(golden[name]["offsets"], golden[name]["indices"], c.cpu().numpy()) == 0
    csr, g, (off, col, _) = s16
    c, _ = ess.color(ctx, g)
    assert np.array_equal(c.cpu().numpy(), oracle.color_jacobi(off, col)[0])


# ------------------------------------------------------------------------------------------------ operators
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


@pytest.mark.parametrize("direction", ["forward", "backward"])
@pytest.mark.parametrize("lb", LBS)
def test_advance_operator_multiset(ctx, lb, direction):
    """Operator-level contract: op runs exactly once per (frontier item, edge) — holes skipped, duplicates
    expanded twice — and the output is exactly the multiset of kept neighbours (order unspecified)."""
    csr = gg.rmat_csr(11, symmetric=False, device="cuda")
    csc = ess.transpose(csr)
    g = ess.Graph(csr, csc=csc)
    view = csr if direction == "forward" else csc
    off, col, _ = view.host()
    rng = np.random.default_rng(5)
    cases = {
        "random+holes+dups": np.concatenate([rng.integers(0, csr.n, 700), -np.ones(40, np.int64),
                                             rng.integers(0, csr.n, 30).repeat(2)]),
        "all": np.arange(csr.n),
        "single-hub": np.array([int(np.argmax(np.diff(off)))]),
        "only-holes": -np.ones(17, np.int64),
        "empty": np.zeros(0, np.int64),
    }
    for label, f in cases.items():
        f = f.astype(np.int32)
        rng.shuffle(f)
        out, calls = ess.advance_probe(ctx, g, torch.from_numpy(f).cuda(), lb=lb, direction=direction, modulus=3)
        want, want_calls = _expected_advance(off, col, f, 3)
        assert np.array_equal(np.sort(out.cpu().numpy()), want), (lb, direction, label)
        assert np.array_equal(calls.cpu().numpy()[: col.size], want_calls[: col.size]), (lb, direction, label)


@pytest.mark.parametrize("lb", LBS)
def test_advance_unique_operator(ctx, lb):
    """operators::advance::execute_unique (fused advance + uniquify, SURVEY §8f row 1): op still runs once per
    (frontier item, edge) — the probe calls it twice, so twice — but the output is the SET of kept neighbours, and
    the second call on the same bitmap reproduces it (the epilogue left the map clear)."""
    csr = gg.rmat_csr(11, symmetric=False, device="cuda")
    g = ess.Graph(csr)
    off, col, _ = csr.host()
    rng = np.random.default_rng(6)
    cases = {
        "random+holes+dups": np.concatenate([rng.integers(0, csr.n, 700), -np.ones(40, np.int64),
                                             rng.integers(0, csr.n, 30).repeat(2)]),
        "all": np.arange(csr.n),
        "single-hub": np.array([int(np.argmax(np.diff(off)))]),
        "only-holes": -np.ones(17, np.int64),
        "empty": np.zeros(0, np.int64),
    }
    for label, f in cases.items():
        f = f.astype(np.int32)
        rng.shuffle(f)
        out, calls = ess.advance_unique_probe(ctx, g, torch.from_numpy(f).cuda(), lb=lb, modulus=3)
        want, want_calls = _expected_advance(off, col, f, 3)
        got = out.cpu().numpy()
        assert np.array_equal(np.sort(got), np.unique(want)), (lb, label)
        assert np.array_equal(calls.cpu().numpy()[: col.size], 2 * want_calls[: col.size]), (lb, label)


@pytest.mark.parametrize("alg", ["predicated", "remove", "compact", "bypass"])
def test_filter_operator(ctx, graphs, alg):
    g = graphs["rmat_s10"]
    rng = np.random.default_rng(9)
    for size in (0, 1, 5, 1023, 1024, 1025, 40000):
        items = rng.integers(0, g.n, size).astype(np.int32)
        items[rng.random(size) < 0.1] = -1
        keep = (items >= 0) & (items % 3 != 0)
        out, calls = ess.filter_probe(ctx, g, torch.from_numpy(items).cuda(), alg=alg, modulus=3)
        got = out.cpu().numpy()
        if alg == "bypass":
            assert np.array_equal(got, np.where(keep, items, -1)), size
        else:
            assert np.array_equal(got, items[keep]), f"{alg} must be a stable compaction (size {size})"
        want_calls = np.bincount(items[items >= 0], minlength=g.n)
        assert np.array_equal(calls.cpu().numpy()[: g.n], want_calls), "op exactly once per valid element"
    items = torch.from_numpy(np.arange(5000, dtype=np.int32) % g.n).cuda()
    out, _ = ess.filter_probe(ctx, g, items, alg="bypass", modulus=3, in_place=True)
    want = np.arange(5000) % g.n
    assert np.array_equal(out.cpu().numpy(), np.where(want % 3 != 0, want, -1))


def test_uniquify_operator(ctx, graphs):
    g = graphs["rmat_s10"]
    rng = np.random.default_rng(4)
    for size in (0, 1, 33, 5000, 70000):
        items = rng.integers(0, g.n, size).astype(np.int32)
        items[rng.random(size) < 0.05] = -1
        out = ess.uniquify_probe(ctx, g, torch.from_numpy(items).cuda())
        assert np.array_equal(out.cpu().numpy(), np.unique(items[items >= 0])), size


def test_frontier_sparse_dense_round_trip(ctx):
    rng = np.random.default_rng(2)
    for universe in (1, 31, 32, 33, 1000, 100003):
        ids = np.unique(rng.integers(0, universe, universe // 3 + 1)).astype(np.int32)
        noisy = np.concatenate([ids, ids[: len(ids) // 2], -np.ones(3, np.int32)])  # duplicates and holes
        words, pop = ess.frontier_to_bitmap(ctx, torch.from_numpy(noisy).cuda(), universe)
        assert pop == ids.size
        bits = np.unpackbits(words.cpu().numpy().view(np.uint8), bitorder="little")[:universe]
        assert np.array_equal(np.nonzero(bits)[0].astype(np.int32), ids)
        back = ess.bitmap_to_frontier(ctx, words, universe)
        assert np.array_equal(np.sort(back.cpu().numpy()), ids)


def test_device_transpose_matches_host_transpose(ctx):
    csr = gg.rmat_csr(12, symmetric=False, weights="hash", device="cuda")
    t = ess.transpose(csr)
    ref = gg.transpose_csr(csr)
    assert torch.equal(t.offsets, ref.offsets)
    key = lambda c: torch.sort(torch.repeat_interleave(torch.arange(c.n, device="cuda"), c.degrees().long()) * c.n
                               + c.indices.long())[0]
    assert torch.equal(key(t), key(ref))
    # weights travel with their edge
    order = lambda c: torch.argsort(torch.repeat_interleave(torch.arange(c.n, device="cuda"), c.degrees().long())
                                    * c.n + c.indices.long())
    assert torch.equal(t.values[order(t)], ref.values[order(ref)])
