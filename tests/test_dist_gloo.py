"""CPU suite: the multi-GPU BFS host logic (1-D partition, bitmap exchange, direction switch, termination) on
world_size 2 and 4 with the gloo backend. The per-rank level kernels are replaced by a numpy stand-in with
the same contract as ess_bfs_partition_step / ess_bfs_partition_pull / ess_bfs_absorb (this double lives in tests/, not the product)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle
from essentials_b200 import dist as edist
from essentials_b200 import graphgen as gg


class NumpyBackend:
    def __init__(self, csr_local, row_begin, n_global):
        self.off = csr_local.offsets.numpy().astype(np.int64)
        self.col = csr_local.indices.numpy()
        self.val = csr_local.values.numpy() if csr_local.values is not None else None
        self.row_begin, self.n_global, self.n_local = row_begin, n_global, self.off.size - 1

    @staticmethod
    def _bits(words, n):
        return np.unpackbits(words.numpy().view(np.uint8), bitorder="little")[:n].astype(bool)

    @staticmethod
    def _store(words, flags, lo_word):
        packed = np.packbits(flags, bitorder="little").view(np.int32)
        words[lo_word:lo_word + packed.size] = torch.from_numpy(packed.copy())

    def pull(self, level, frontier_bits, visited_bits, next_slice, depth_local, counts):
        n, lo = self.n_global, self.row_begin
        frontier, visited = self._bits(frontier_bits, n), self._bits(visited_bits, n)
        found = np.zeros(self.n_local, bool)
        for v in range(self.n_local):
            if not visited[lo + v]:
                nb = self.col[self.off[v]:self.off[v + 1]]
                found[v] = frontier[nb].any()
        ids = np.nonzero(found)[0]
        depth_local[torch.from_numpy(ids)] = level
        visited[lo:lo + self.n_local] |= found
        self._store(visited_bits, visited, 0)
        self._store(next_slice, found, 0)
        counts.view(torch.int64)[0] += int(found.sum())  # counts[1] untouched, as ess_bfs_partition_pull

    def merge(self, gathered, world, slice_words, frontier_bits, visited_bits, counts_out):
        rows = gathered.view(world, slice_words + 4)
        frontier_bits.view(world, slice_words).copy_(rows[:, :slice_words])
        visited_bits[: world * slice_words].bitwise_or_(frontier_bits)
        counts_out.copy_(rows[:, slice_words:].contiguous().view(torch.int64).reshape(-1))

    def gather_fresh(self, next_slice, fresh_list):
        ids = np.nonzero(self._bits(next_slice, self.n_local))[0]
        fresh_list[: ids.size] = torch.from_numpy(ids.astype(np.int32))

    def step(self, pull, frontier_bits, visited_bits, candidate_bits, frontier_list, frontier_count):
        n, lo = self.n_global, self.row_begin
        frontier, visited = self._bits(frontier_bits, n), self._bits(visited_bits, n)
        assert not pull
        if False:
            pass
        else:
            cand = np.zeros(n, bool)
            mine = frontier_list.numpy()[:frontier_count]
            assert sorted(mine.tolist()) == np.nonzero(frontier[lo:lo + self.n_local])[0].tolist(), \
                "sparse list and frontier bitmap of a rank must describe the same set"
            for v in mine:
                nb = self.col[self.off[v]:self.off[v + 1]]
                cand[nb[~visited[nb]]] = True
            self._store(candidate_bits, cand, 0)

    def absorb(self, level, candidates, n_slices, stride_words, visited_bits, next_slice, depth_local, fresh_list,
               counts):
        n, lo = self.n_global, self.row_begin
        c = candidates.numpy()
        words = np.zeros((self.n_local + 31) // 32, np.int32)
        for p in range(n_slices):
            words |= c[p * stride_words:p * stride_words + words.size]
        cand = np.unpackbits(words.view(np.uint8), bitorder="little")[: self.n_local].astype(bool)
        visited = self._bits(visited_bits, n)
        fresh = cand & ~visited[lo:lo + self.n_local]
        ids = np.nonzero(fresh)[0]
        depth_local[torch.from_numpy(ids)] = level
        fresh_list[: ids.size] = torch.from_numpy(ids.astype(np.int32))
        visited[lo:lo + self.n_local] |= fresh
        self._store(visited_bits, visited, 0)
        self._store(next_slice, fresh, 0)
        deg = np.diff(self.off)
        counts.view(torch.int64)[0] += int(fresh.sum())
        counts.view(torch.int64)[1] += int(deg[fresh].sum())


    # ---- SSSP stand-ins (contract of ess_sssp_partition_relax / ess_sssp_partition_collect) ----
    def relax(self, active_list, active_count, dist_local, replica):
        rep, d = replica.numpy(), dist_local.numpy()
        for v in active_list.numpy()[:active_count]:
            lo, hi = self.off[v], self.off[v + 1]
            cand = (d[v] + self.val[lo:hi]).astype(np.float32)  # float32 add, as the device does
            np.minimum.at(rep, self.col[lo:hi], cand)

    def collect(self, reduced, dist_local, active_list, counts):
        r, d = reduced.numpy(), dist_local.numpy()
        ids = np.nonzero(r < d)[0]
        d[ids] = r[ids]
        active_list[: ids.size] = torch.from_numpy(ids.astype(np.int32))
        counts[0] += int(ids.size)
        counts[1] += int(np.diff(self.off)[ids].sum())


def _sssp_worker(rank, world, port, scale, sources, out):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        n = 1 << scale
        per = n // world
        csr = gg.rmat_csr(scale, row_range=(rank * per, (rank + 1) * per), weights="hash")
        runner = edist.PartitionedSSSP(csr, rank * per, n, rank, world, NumpyBackend(csr, rank * per, n),
                                       torch.device("cpu"))
        results = {}
        for s in sources:
            info = runner.sssp(s)
            results[s] = (runner.gather_dist().numpy().copy(), info, runner.reached_work())
        if rank == 0:
            out.put(results)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])
def test_partitioned_sssp_matches_oracle(world):
    scale = 9
    full = gg.rmat_csr(scale, weights="hash")
    off, col, val = full.host()
    sources = [0, int(torch.nonzero(full.degrees() == 0)[0])] + gg.pick_sources(full, 2)
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_sssp_worker, args=(r, world, port, scale, sources, out)) for r in range(world)]
    for p in procs:
        p.start()
    results = out.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    deg = np.diff(off)
    for s, (got, info, (n_r, m_r)) in results.items():
        want = oracle.sssp(off, col, val, s)
        assert np.array_equal(got, want), f"source {s}"  # bit-exact: unique fixed point of float32 min-plus
        reached = want != np.float32(3.4028234663852886e38)
        assert n_r == int(reached.sum()) and m_r == int(deg[reached].sum())
        assert info["iterations"] >= 1 and info["relaxed_edges"] >= m_r - int(deg[s] == 0)


def _worker(rank, world, port, scale, sources, out):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        n = 1 << scale
        per = n // world
        csr = gg.rmat_csr(scale, row_range=(rank * per, (rank + 1) * per))
        runner = edist.PartitionedBFS(csr, rank * per, n, rank, world, NumpyBackend(csr, rank * per, n),
                                      torch.device("cpu"))
        picks = runner.pick_sources(3)
        results = {}
        for s in sources + picks:
            info = runner.bfs(s)
            results[s] = (runner.gather_depth().numpy().copy(), info, runner.reached_work())
        if rank == 0:
            out.put((picks, {k: (v[0], v[1], v[2]) for k, v in results.items()}))
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("world", [2, 4])
def test_partitioned_bfs_matches_oracle(world):
    scale = 10
    full = gg.rmat_csr(scale)
    off, col, _ = full.host()
    fixed = [0, int(torch.nonzero(full.degrees() == 0)[0])]  # the reference driver's source 0, and an isolated one
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, _free_port() if r == 0 else 0, scale, fixed, out))
             for r in range(world)]
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, scale, fixed, out)) for r in range(world)]
    for p in procs:
        p.start()
    picks, results = out.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert picks == gg.pick_sources(full, 3), "distributed source picking must agree with the single-GPU one"
    deg = np.diff(off)
    saw_pull = False
    for s, (depth, info, (n_r, m_r)) in results.items():
        want = oracle.bfs(off, col, s)
        assert np.array_equal(depth, want), f"source {s}"
        assert n_r == int((want != 2**31 - 1).sum()) and m_r == int(deg[want != 2**31 - 1].sum())
        assert info["iterations"] == int(want[want != 2**31 - 1].max()) + 1
        saw_pull |= info["pull_steps"] > 0
    assert saw_pull, "the Kronecker graph must exercise the bottom-up exchange path"


def test_pack_bits_round_trip():
    rng = np.random.default_rng(0)
    flags = rng.random(32 * 37) < 0.3
    words = edist._pack_bits(torch.from_numpy(flags))
    back = np.unpackbits(words.numpy().view(np.uint8), bitorder="little").astype(bool)
    assert np.array_equal(back, flags)
    assert edist._bit(31) == -(2**31) and edist._bit(0) == 1
