"""CPU suite: the betweenness-centrality contract (include/essentials_b200.h, ess_bc) as the tests restate it, and the
host-side argument checks of ess.bc.

bc_ref.brandes (the float64 restatement the GPU tests compare against) must equal bc_ref.brute_force, which counts
shortest paths straight from the definition, on small directed and symmetric multigraphs with self-loops, parallel
edges and several components. The certificate the GPU tests and scripts/bc_cost.py check on large graphs,
Σ_{v != s} δ_s(v) == Σ_{t reached, t != s} (depth[t] - 1), is checked here on the restatement."""
import types

import numpy as np
import pytest
import torch

import bc_ref as ref
import essentials_b200 as ess


@pytest.mark.parametrize("symmetric", [False, True])
def test_brandes_restatement_equals_the_definition(symmetric):
    rng = np.random.default_rng(97 + symmetric)
    checked = parallel = loops = split = 0
    for _ in range(60):
        n, src, dst = ref.random_multigraph(rng, symmetric)
        off, col = ref.from_edges(n, src, dst)
        want = ref.brute_force(off, col)
        assert np.allclose(ref.brandes(off, col), want, rtol=1e-12, atol=1e-12)
        sub = [int(x) for x in rng.integers(0, n, 3)]
        assert np.allclose(ref.brandes(off, col, sub), ref.brute_force(off, col, sub), rtol=1e-12, atol=1e-12)
        pairs = src * n + dst
        parallel += np.unique(pairs).size < pairs.size
        loops += bool((src == dst).any())
        split += int((ref.depths(n, *ref.edge_list(off, col), 0) < 0).any())
        checked += 1
    assert checked == 60 and parallel and loops and split  # the cases the contract names all occurred


def test_parallel_edges_are_distinct_paths_and_self_loops_never_count():
    """0 -> 1 twice, 0 -> 2, 1 -> 3, 2 -> 3, 3 -> 3: three shortest 0 -> 3 paths, two of them through 1."""
    off, col = ref.from_edges(4, [0, 0, 0, 1, 2, 3], [1, 1, 2, 3, 3, 3])
    bc = ref.brandes(off, col, [0])
    assert np.allclose(bc, [0.0, 2.0 / 3.0, 1.0 / 3.0, 0.0])
    assert np.allclose(ref.brute_force(off, col, [0]), bc)


def test_scale_and_repeated_sources():
    rng = np.random.default_rng(5)
    n, src, dst = ref.random_multigraph(rng, True)
    off, col = ref.from_edges(n, src, dst)
    one = ref.brandes(off, col, [0])
    assert np.array_equal(ref.brandes(off, col, [0, 0]), 2 * one)
    assert np.array_equal(ref.brandes(off, col, [0], scale=0.5), 0.5 * one)


def test_sum_of_dependencies_certificate():
    rng = np.random.default_rng(11)
    for symmetric in (False, True):
        for _ in range(30):
            n, src, dst = ref.random_multigraph(rng, symmetric)
            off, col = ref.from_edges(n, src, dst)
            rows, cols = ref.edge_list(off, col)
            for s in range(n):
                delta, depth = ref.dependencies(n, rows, cols, s)
                reached = depth > 0
                assert np.isclose(delta.sum() - delta[s], (depth[reached] - 1).sum(), rtol=1e-12, atol=1e-12)
                assert delta.min() >= 0


# ----------------------------------------------------------------------------------- ess.bc host-side checks
def _fake(n=10):
    """A context and graph that only carry what ess.bc reads before it calls the library."""
    return types.SimpleNamespace(handle=None), types.SimpleNamespace(n=n, handle=None, has_csc=True,
                                                                     device=torch.device("cuda", 0))


@pytest.mark.parametrize("sources, match", [
    (-1, "out of range"), (10, "out of range"), ([0, 3, 10], "out of range"), ([], "empty"),
    ([1.0], "vertex ids"), ([True], "vertex ids"), ("3", "vertex ids"), (2.0, "vertex ids"),
    (torch.tensor([1.0]), "CPU integer tensor"), (torch.tensor([0, 12]), "out of range"),
])
def test_bc_rejects_bad_sources_without_a_device(sources, match):
    ctx, g = _fake()
    with pytest.raises(ess.EssentialsError, match=match):
        ess.bc(ctx, g, sources)


@pytest.mark.parametrize("scale", [float("nan"), float("inf"), -float("inf")])
def test_bc_rejects_non_finite_scale_without_a_device(scale):
    ctx, g = _fake()
    with pytest.raises(ess.EssentialsError, match="finite"):
        ess.bc(ctx, g, [1], scale=scale)


@pytest.mark.parametrize("out", [torch.zeros(10, dtype=torch.float32), np.zeros(10, np.float32)])
def test_bc_rejects_an_out_buffer_off_the_device(out):
    ctx, g = _fake()
    with pytest.raises(ess.EssentialsError, match="float32 CUDA tensor"):
        ess.bc(ctx, g, [1, 2], out=out)
