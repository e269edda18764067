"""CPU suite: the SSSP tree contract (include/essentials_b200.h, ess_sssp_tree) as the tests restate it.

sssp_tree_ref (a plain C++ restatement, the reference the GPU tests compare against) must equal an independent numpy
restatement of rules 1-4 on arbitrary directed multigraphs, its trees must be valid (source, unreached, tight parent
edges, no cycles), and every kind of forged distance array must return its own violation code. The torch checker
scripts/sssp_tree_cost.py uses on the device runs here on host tensors: each of its rules must fire on a tree broken in
exactly that way."""
import importlib.util
import os

import numpy as np
import torch

import oracle
import sssp_tree_ref as ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FMAX = np.float32(np.finfo(np.float32).max)
NONE = np.iinfo(np.int32).max


def _load_cost_script():
    spec = importlib.util.spec_from_file_location("sssp_tree_cost", os.path.join(ROOT, "scripts", "sssp_tree_cost.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


sssp_tree_violations = _load_cost_script().sssp_tree_violations


def from_edges(n, src, dst, w):
    order = np.lexsort((dst, src))
    off = np.zeros(n + 1, np.int64)
    np.add.at(off, np.asarray(src) + 1, 1)
    return np.cumsum(off), np.asarray(dst, np.int32)[order], np.asarray(w, np.float32)[order]


WEIGHTS = np.array([0.0, 0.0, 0.5, 1.0, 1.0, 2.25, 7.0, 1e8, 3e8], np.float32)


def arbitrary_multigraph(rng):
    """Directed multigraph with self loops, parallel edges, isolated vertices, zero weights, and weights that rounding
    absorbs next to 1e8 (fl(1e8 + w) == 1e8 for w <= 4)."""
    n = int(rng.integers(2, 60))
    m = int(rng.integers(1, 300))
    return (n,) + from_edges(n, rng.integers(0, n, m), rng.integers(0, n, m), rng.choice(WEIGHTS, m))


def numpy_tree(off, col, w, s, d):
    """Rules 1-4, vectorised over the edge list. Returns (pred, flat rounds)."""
    n = off.size - 1
    rows = np.repeat(np.arange(n), np.diff(off))
    col = col.astype(np.int64)
    w = np.ones(col.size, np.float32) if w is None else w
    du, dv = d[rows], d[col]
    through = (du + w).astype(np.float32)
    tight = (du < FMAX) & (through == dv)
    strict = tight & (du < dv)
    flat = tight & (du == dv) & (rows != col)
    pred = np.full(n, NONE, np.int64)
    np.minimum.at(pred, col[strict], rows[strict])
    pred[s] = s
    reached = d < FMAX
    level = np.where(reached & (pred != NONE), 0, -1)
    fr, fc = rows[flat], col[flat]
    k = 0
    while True:
        step = (level[fr] == k) & (level[fc] == -1)
        if not step.any():
            break
        k += 1
        cand = np.full(n, NONE, np.int64)
        np.minimum.at(cand, fc[step], fr[step])
        new = cand != NONE
        pred[new], level[new] = cand[new], k
    assert not (reached & (level == -1)).any(), "a reached vertex without a parent"
    pred[~reached] = -1
    return pred.astype(np.int32), k


def check_tree(off, col, w, s, d, pred):
    """Validity on host arrays: source, unreached, tight parent edge, every chain ends at the source."""
    n = off.size - 1
    assert pred[s] == s
    reached = d < FMAX
    assert np.array_equal(pred == -1, ~reached)
    w = np.ones(col.size, np.float32) if w is None else w
    tight_edges = set()
    for u in range(n):
        for e in range(off[u], off[u + 1]):
            if d[u] < FMAX and np.float32(d[u] + w[e]) == d[col[e]]:
                tight_edges.add((u, int(col[e])))
    for v in np.flatnonzero(reached):
        if v != s:
            assert (int(pred[v]), int(v)) in tight_edges, ("parent edge not tight", v, pred[v])
        x, hops = int(v), 0
        while x != s:
            x, hops = int(pred[x]), hops + 1
            assert hops <= n, ("cycle through", v)


def test_reference_equals_numpy_restatement_on_arbitrary_multigraphs():
    rng = np.random.default_rng(41)
    deepest, absorbed = 0, 0
    for trial in range(400):
        n, off, col, w = arbitrary_multigraph(rng)
        for s in {0, int(rng.integers(0, n)), n - 1}:
            d = oracle.sssp(off, col, w, s)
            pred, status = ref.sssp_tree(off, col, w, s, d)
            assert status == ref.OK, (trial, s, ref.STATUS[status])
            want, rounds = numpy_tree(off, col, w, s, d)
            assert np.array_equal(pred, want), (trial, s)
            check_tree(off, col, w, s, d, pred)
            deepest = max(deepest, rounds)
            rows = np.repeat(np.arange(n), np.diff(off))
            absorbed += int(((w > 0) & (d[rows] < FMAX) & (d[rows] == d[col]) & (rows != col)).sum())
    assert deepest >= 2 and absorbed > 0, (deepest, absorbed)


def test_unweighted_graph_uses_weight_one():
    n, off, col, _ = arbitrary_multigraph(np.random.default_rng(42))
    d = oracle.sssp(off, col, np.ones(col.size, np.float32), 0)
    pred, status = ref.sssp_tree(off, col, None, 0, d)
    assert status == ref.OK
    assert np.array_equal(pred, numpy_tree(off, col, None, 0, d)[0])


def forged_graph():
    """0 -1-> 1 -0-> 2 -2-> 3, 0 -5-> 3, 3 <-0-> 4 (a reachable zero-weight cycle), 2 -4-> 7 (a leaf), and 5 <-0-> 6
    (a zero-weight cycle the source does not reach)."""
    edges = [(0, 1, 1), (1, 2, 0), (2, 3, 2), (0, 3, 5), (3, 4, 0), (4, 3, 0), (5, 6, 0), (6, 5, 0), (2, 7, 4)]
    src, dst, w = zip(*edges)
    return from_edges(8, src, dst, w)


def forged_distances():
    """{case: (distances, expected status)} on forged_graph() from source 0."""
    off, col, w = forged_graph()
    d = oracle.sssp(off, col, w, 0)
    assert d.tolist() == [0, 1, 1, 3, 3, FMAX, FMAX, 5]
    cases = {}

    def forge(name, at, value, status):
        x = d.copy()
        x[at] = value
        cases[name] = (x, status)

    forge("lowered", 7, 4.5, ref.ORPHAN)
    forge("raised", 2, 1.5, ref.RELAXABLE_EDGE)
    forge("source not 0", 0, 1.0, ref.SOURCE_NOT_ZERO)
    forge("NaN", 4, np.nan, ref.INVALID_ENTRY)
    forge("negative", 7, -1.0, ref.INVALID_ENTRY)
    forge("infinite", 5, np.inf, ref.INVALID_ENTRY)
    forge("reached vertex marked FLT_MAX", 3, FMAX, ref.RELAXABLE_EDGE)
    x = d.copy()
    x[[5, 6]] = 7.0
    cases["unreachable zero-weight cycle"] = (x, ref.ORPHAN)
    return cases


def test_forged_distances_return_their_violation():
    off, col, w = forged_graph()
    d = oracle.sssp(off, col, w, 0)
    pred, status = ref.sssp_tree(off, col, w, 0, d)
    assert status == ref.OK
    assert pred.tolist() == [0, 0, 1, 2, 3, -1, -1, 2]
    for name, (x, want) in forged_distances().items():
        assert ref.sssp_tree(off, col, w, 0, x)[1] == want, name


def test_device_checker_accepts_valid_trees_on_host_tensors():
    rng = np.random.default_rng(43)
    for trial in range(40):
        n, off, col, w = arbitrary_multigraph(rng)
        s = int(rng.integers(0, n))
        d = oracle.sssp(off, col, w, s)
        pred, status = ref.sssp_tree(off, col, w, s, d)
        assert status == ref.OK
        got = sssp_tree_violations(torch.from_numpy(off), torch.from_numpy(col), torch.from_numpy(w), s,
                                   torch.from_numpy(d), torch.from_numpy(pred), chunk=64)
        assert not any(got.values()), (trial, got)


def test_device_checker_finds_each_broken_rule():
    off, col, w = forged_graph()
    d = oracle.sssp(off, col, w, 0)
    pred, _ = ref.sssp_tree(off, col, w, 0, d)
    args = (torch.from_numpy(off), torch.from_numpy(col), torch.from_numpy(w), 0, torch.from_numpy(d))
    assert not any(sssp_tree_violations(*args, torch.from_numpy(pred), chunk=4).values())
    broken = {"source": {0: -1}, "unreached": {7: -1}, "range": {7: 8}, "edge": {7: 1},  # 1 -> 7: no such edge
              "cycle": {3: 4}}  # 3 <-> 4: both edges tight, neither reaches the source
    for rule, changes in broken.items():
        p = pred.copy()
        for at, value in changes.items():
            p[at] = value
        got = sssp_tree_violations(*args, torch.from_numpy(p), chunk=4)
        assert got[rule] > 0, (rule, got)
    # a parent edge that exists but is not tight: 0 -> 3 has weight 5, d[3] == 3
    p = pred.copy()
    p[3] = 0
    assert sssp_tree_violations(*args, torch.from_numpy(p), chunk=4)["edge"] == 1

