"""CPU suite: the k-core oracle (oracle/oracle.cpp, the reference's peel restated) against the textbook definition —
the core number of v is the largest k such that v lies in the k-core, the largest subgraph whose minimum degree is at
least k — on simple symmetric graphs, where the two definitions coincide. Also: the entry points that write one label
per vertex refuse an `out=` that is not a CUDA tensor before they call the library. No GPU."""
import types

import numpy as np
import pytest
import torch

import essentials_b200 as ess
import oracle
from essentials_b200 import graphgen as gg


def textbook_core_numbers(off, col):
    """For k = 1, 2, ...: delete vertices of degree < k until none is left (the k-core remains); core(v) = the last k
    whose k-core still holds v. Written from the definition, independently of the oracle's peel order."""
    off, col = np.asarray(off, np.int64), np.asarray(col, np.int64)
    n = off.size - 1
    rows = np.repeat(np.arange(n), np.diff(off))
    core = np.zeros(n, np.int32)
    alive = np.diff(off) > 0
    k = 0
    while alive.any():
        k += 1
        while True:
            live = alive[rows] & alive[col]
            deg = np.bincount(rows[live], minlength=n)
            drop = alive & (deg < k)
            if not drop.any():
                break
            alive &= ~drop
        core[alive] = k
    return core


def _simple(n, u, v):
    """Simple symmetric CSR (no self-loops, no parallel edges) of the undirected edges (u, v)."""
    u, v = np.asarray(u, np.int64), np.asarray(v, np.int64)
    keep = u != v
    key = np.unique(np.concatenate([u[keep] * n + v[keep], v[keep] * n + u[keep]]))
    off = np.zeros(n + 1, np.int64)
    np.add.at(off, key // n + 1, 1)
    return np.cumsum(off), (key % n).astype(np.int32)


RANDOM_TRIALS = 12
CASES = ["K_9 plus a pendant path", "cycle and path", "star with a triangle at its centre", "grid 12x9",
         *[f"random {t}" for t in range(RANDOM_TRIALS)], "rmat 8", "rmat 11", "rmat 12"]


def _case(name):
    if name == "K_9 plus a pendant path":
        a, b = np.triu_indices(9, 1)
        return _simple(13, np.r_[a, 8:12], np.r_[b, 9:13])
    if name == "cycle and path":  # 0..8 a cycle, 9..18 a path, 19 isolated
        return _simple(20, np.r_[0:9, 9:18], np.r_[(np.arange(9) + 1) % 9, 10:19])
    if name == "star with a triangle at its centre":  # centre 0, leaves 1..57, the edge 1-2 closes a triangle
        return _simple(60, np.r_[np.zeros(57, np.int64), 1], np.r_[1:58, 2])
    if name == "grid 12x9":
        return gg.grid_csr(12, 9).host()[:2]
    if name.startswith("random"):
        rng = np.random.default_rng(int(name.split()[1]))
        n = int(rng.integers(5, 300))
        m = int(rng.integers(0, 6 * n))
        return _simple(n, rng.integers(0, n, m), rng.integers(0, n, m))
    return gg.rmat_csr(int(name.split()[1])).host()[:2]


@pytest.mark.parametrize("name", CASES)
def test_kcore_oracle_is_the_textbook_core_number(name):
    off, col = _case(name)
    want = textbook_core_numbers(off, col)
    assert np.array_equal(oracle.kcore(off, col), want), name


def test_textbook_core_numbers_on_known_graphs():
    """The definition above on answers that can be written down: K_9 has core 8 and its pendant path core 1; a cycle
    core 2, a path core 1, an isolated vertex 0; a star's leaves core 1, its centre core 2 when it lies on a triangle;
    a grid core 2."""
    assert textbook_core_numbers(*_case("K_9 plus a pendant path")).tolist() == [8] * 9 + [1] * 4
    assert textbook_core_numbers(*_case("cycle and path")).tolist() == [2] * 9 + [1] * 10 + [0]
    assert textbook_core_numbers(*_case("star with a triangle at its centre")).tolist() == [2] * 3 + [1] * 55 + [0] * 2
    assert textbook_core_numbers(*_case("grid 12x9")).tolist() == [2] * 108


OUT_DTYPES = {"bfs": torch.int32, "sssp": torch.float32, "sssp_near_far": torch.float32, "sssp_delta": torch.float32,
              "pagerank": torch.float32, "ppr": torch.float32, "kcore": torch.int32, "color": torch.int32}


def _call(entry, ctx, g, out):
    if entry in ("bfs", "sssp", "sssp_near_far", "sssp_delta", "ppr"):
        return getattr(ess, entry)(ctx, g, 0, out=out)
    return getattr(ess, entry)(ctx, g, out=out)


@pytest.mark.parametrize("entry", list(OUT_DTYPES))
def test_out_off_the_device_is_refused_without_a_device(entry):
    """A host tensor of the right dtype and size, and a numpy array: refused by the binding, not handed to a kernel."""
    ctx = types.SimpleNamespace(handle=None)
    g = types.SimpleNamespace(n=10, handle=None, has_csc=True, device=torch.device("cuda", 0))
    dtype = OUT_DTYPES[entry]
    name = str(dtype).replace("torch.", "")
    for out in (torch.zeros(10, dtype=dtype), np.zeros(10, np.int32 if dtype == torch.int32 else np.float32)):
        with pytest.raises(ess.EssentialsError, match=f"contiguous {name} CUDA tensor of at least 10 elements"):
            _call(entry, ctx, g, out)
