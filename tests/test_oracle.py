"""CPU suite: pins the oracle restatement (oracle/oracle.cpp) against (1) the committed known-answer vectors
the reference's own CPU code produced (tests/golden, SURVEY.md §4) and (2) that reference code itself when
oracle/_ref was built here, or else its stored outputs on the same inputs. No GPU, no CUDA library compute."""
import os

import numpy as np
import pytest

import oracle
from essentials_b200 import graphgen

# the reference's outputs on the inputs of the two tests below that run its code (tests/golden/make_reference_vectors.py)
STORED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.npz")

SURVEY_BFS = "0 2 2 2 2 2 1 1 2 2 1 1 1 2 2 2 2 2 2 2 2 1 1 2 2 2 2 2 2 2 2 2 2 1 1 2 1 2 1"
SURVEY_KCORE = "6 6 5 3 3 3 6 6 6 5 6 6 6 6 6 5 3 6 6 4 5 6 6 4 6 6 6 6 6 6 5 6 6 3 6 6 3 6 6"


def test_survey_known_answers(golden):
    g = golden["chesapeake"]
    off, col, val = g["offsets"], g["indices"], g["values"]
    assert off.size - 1 == 39 and col.size == 340
    want_bfs = np.array(SURVEY_BFS.split(), np.int32)
    assert np.array_equal(oracle.bfs(off, col, 0), want_bfs)
    assert np.array_equal(oracle.sssp(off, col, val, 0), want_bfs.astype(np.float32))
    assert np.array_equal(oracle.kcore(off, col), np.array(SURVEY_KCORE.split(), np.int32))
    p = oracle.ppr(off, col, 0)
    assert abs(float(p.sum()) - 0.9997149664) < 1e-6
    assert np.allclose(p[:5], [0.296592623, 0.02544574253, 0.005980789196, 0.009085948579, 0.01279114652], atol=1e-7)


@pytest.mark.parametrize("name", ["chesapeake", "rmat_s10", "grid_24x17"])
def test_oracle_matches_golden(golden, name):
    g = golden[name]
    off, col, val = g["offsets"], g["indices"], g["values"]
    for s in g["sources"]:
        assert np.array_equal(oracle.bfs(off, col, int(s)), g[f"bfs_{s}"]), f"bfs from {s}"
        assert np.array_equal(oracle.sssp(off, col, val, int(s)), g[f"sssp_{s}"]), f"sssp from {s} (bit-exact)"
    assert np.array_equal(oracle.kcore(off, col), g["kcore"])
    for s in g["ppr_seeds"]:
        assert np.array_equal(oracle.ppr(off, col, int(s)), g[f"ppr_{s}"]), "ppr restatement is bit-exact on CPU"
    n = off.size - 1
    assert np.array_equal(oracle.randoms(n, 0.0, float(n)), g["randoms"])


def test_color_oracle_is_valid_and_deterministic(golden):
    for name in ("chesapeake", "rmat_s10", "grid_24x17"):
        g = golden[name]
        off, col = g["offsets"], g["indices"]
        c1, it1 = oracle.color_jacobi(off, col, g["randoms"])
        c2, it2 = oracle.color_jacobi(off, col)
        assert np.array_equal(c1, c2) and it1 == it2
        assert oracle.color_errors(off, col, c1) == 0
        assert c1.min() >= 0 and c1.max() < 2 * it1


def test_pagerank_oracle_properties(golden):
    g = golden["rmat_s10"]
    off, col, val = g["offsets"], g["indices"], g["values"]
    p, it = oracle.pagerank(off, col, np.ones_like(val))
    assert 1 < it < 200
    assert abs(float(p.astype(np.float64).sum()) - 1.0) < 1e-4  # rank mass is conserved (dangling mass re-spread)
    p2, it2 = oracle.pagerank(off, col, np.ones_like(val), force_iters=it)
    assert it2 == it and np.array_equal(p, p2)
    # weights scale out of PageRank: iweights normalise them
    p3, _ = oracle.pagerank(off, col, 3.0 * np.ones_like(val), force_iters=it)
    assert np.allclose(p, p3, rtol=1e-6)


def test_oracle_matches_reference_code_on_fresh_graphs():
    if not oracle.have_ref():
        ref = np.load(STORED)
        for scale, seed in ((8, 3), (11, 5), (12, 1)):
            g = graphgen.rmat_csr(scale, seed=seed, weights="hash")
            off, col, val = g.host()
            sources = graphgen.pick_sources(g, 2, seed=seed)
            assert sources == ref[f"rmat{scale}_sources"].tolist()
            for s in sources:
                assert np.array_equal(oracle.bfs(off, col, s), ref[f"rmat{scale}_bfs_{s}"])
                assert np.array_equal(oracle.sssp(off, col, val, s), ref[f"rmat{scale}_sssp_{s}"])
            assert np.array_equal(oracle.kcore(off, col), ref[f"rmat{scale}_kcore"])
        off, col, val = graphgen.grid_csr(40, 31).host()
        assert np.array_equal(oracle.sssp(off, col, val, 5), ref["grid40x31_sssp_5"])
        return  # PPR, the random stream and colouring need the reference's code itself
    for scale, seed in ((8, 3), (11, 5), (12, 1)):
        g = graphgen.rmat_csr(scale, seed=seed, weights="hash")
        off, col, val = g.host()
        for s in graphgen.pick_sources(g, 2, seed=seed):
            assert np.array_equal(oracle.bfs(off, col, s), oracle.ref_bfs(off, col, s))
            assert np.array_equal(oracle.sssp(off, col, val, s), oracle.ref_sssp(off, col, val, s))
        assert np.array_equal(oracle.kcore(off, col), oracle.ref_kcore(off, col))
        assert np.array_equal(oracle.ppr(off, col, 1), oracle.ref_ppr(off, col, 2)[1])
    g = graphgen.grid_csr(40, 31)
    off, col, val = g.host()
    assert np.array_equal(oracle.sssp(off, col, val, 5), oracle.ref_sssp(off, col, val, 5))
    assert np.array_equal(oracle.randoms(5000, 0.0, 5000.0), oracle.ref_randoms(5000, 0.0, 5000.0))
    # the reference's own colouring (Gauss-Seidel order) is only checked for validity, like color.cu does
    assert oracle.color_errors(off, col, oracle.ref_color(off, col)) == 0


def test_empty_and_degenerate_inputs():
    off = np.array([0, 0, 0, 0], np.int64)  # 3 isolated vertices
    col = np.zeros(0, np.int32)
    assert np.array_equal(oracle.bfs(off, col, 1), [2**31 - 1, 0, 2**31 - 1])
    assert np.array_equal(oracle.kcore(off, col), [0, 0, 0])
    c, it = oracle.color_jacobi(off, col)
    assert np.array_equal(c, [0, 0, 0]) and it == 1
    # a self loop and a multi-edge must not break anything
    off = np.array([0, 3, 4], np.int64)
    col = np.array([0, 1, 1, 0], np.int32)
    assert np.array_equal(oracle.bfs(off, col, 0), [0, 1])
    d = oracle.sssp(off, col, np.array([1, 5, 2, 1], np.float32), 0)
    assert np.array_equal(d, np.array([0, 2], np.float32))


def test_oracle_matches_reference_code_on_arbitrary_small_graphs():
    """Property test (hypothesis): arbitrary small directed multigraphs — self loops, parallel edges, isolated and
    unreachable vertices, equal and zero weights — through the restatement and through the reference's own CPU code.
    Without the reference's code: a fixed set of such multigraphs against the reference's stored outputs."""
    if not oracle.have_ref():
        ref = np.load(STORED)
        count = len([k for k in ref.files if k.startswith("mg") and k.endswith("_bfs")])
        assert count >= 100
        for i in range(count):
            off, col, val = ref[f"mg{i}_offsets"], ref[f"mg{i}_indices"], ref[f"mg{i}_values"]
            s = int(ref[f"mg{i}_source"])
            assert np.array_equal(oracle.bfs(off, col, s), ref[f"mg{i}_bfs"]), i
            assert np.array_equal(oracle.sssp(off, col, val, s), ref[f"mg{i}_sssp"]), i
        return
    from hypothesis import given, settings, strategies as st

    @st.composite
    def graphs(draw):
        n = draw(st.integers(1, 24))
        m = draw(st.integers(0, 80))
        src = draw(st.lists(st.integers(0, n - 1), min_size=m, max_size=m))
        dst = draw(st.lists(st.integers(0, n - 1), min_size=m, max_size=m))
        # dyadic weights (exact in float32) incl. zero and repeats: ties and zero-length edges are the hard cases
        w = draw(st.lists(st.sampled_from([0.0, 0.5, 1.0, 1.0, 2.25, 7.0, 63.984375]), min_size=m, max_size=m))
        order = np.lexsort((np.array(dst, np.int64), np.array(src, np.int64))) if m else np.zeros(0, np.int64)
        s = np.array(src, np.int64)[order]
        off = np.zeros(n + 1, np.int64)
        np.add.at(off, s + 1, 1)
        off = np.cumsum(off)
        return off, np.array(dst, np.int32)[order], np.array(w, np.float32)[order], draw(st.integers(0, n - 1))

    @settings(max_examples=150, deadline=None)
    @given(graphs())
    def check(g):
        off, col, val, s = g
        assert np.array_equal(oracle.bfs(off, col, s), oracle.ref_bfs(off, col, s))
        assert np.array_equal(oracle.sssp(off, col, val, s), oracle.ref_sssp(off, col, val, s))

    check()
