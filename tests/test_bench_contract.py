"""CPU suite: bench.py's contract where it can be exercised without a GPU — the reference arm (`--impl reference`,
the reference's own bfs_cpu from oracle/_ref, or the oracle port) prints ONE JSON line with the agreed keys, and
the product arm refuses to run without a CUDA device instead of falling back to anything on the CPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--scale", "12",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-1500:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "BFS GTEPS" and d["unit"] == "GTEPS"
    for key in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert "workload" in d["config"] and d["value"] > 0 and d["gpu_launches"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and 1 <= cb["cores"] <= 2 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "GTEPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # same `config` object as the product arm prints for this workload (the driver compares them)
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.workload_config(12, 16, d["config"]["n"], d["config"]["m"], 2)
    assert d["scaling"] == "strong"


def _bench_dump(tmp_path, run, *flags):
    """Runs bench.py at scale 12 with --dump-outputs; returns (JSON line, dumped depth array, last timed source)."""
    sys.path.insert(0, ROOT)
    import numpy as np
    from essentials_b200 import graphgen as gg
    out_dir = str(tmp_path / f"dump{run}")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--scale", "12", "--steps", "3", "--warmup",
                          "1", "--dump-outputs", out_dir, *flags], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-1500:]
    assert sorted(os.listdir(out_dir)) == ["bfs_depth.npy"], "4096 vertices are below the sampling threshold"
    depth = np.load(os.path.join(out_dir, "bfs_depth.npy"))
    src = gg.pick_sources(gg.rmat_csr(12, 16), 4)[-1]
    return json.loads(out.stdout.strip().splitlines()[-1]), depth, src


def test_reference_arm_dumps_the_last_timed_bfs(tmp_path):
    """--dump-outputs: the depths of the last timed source, float64, identical from run to run."""
    import numpy as np
    import oracle
    from essentials_b200 import graphgen as gg
    d, depth, src = _bench_dump(tmp_path, 0, "--impl", "reference")
    assert d["steps"] == 3 and depth.dtype == np.float64
    off, col, _ = gg.rmat_csr(12, 16).host()
    assert np.array_equal(depth, oracle.bfs(off, col, src).astype(np.float64))
    assert np.array_equal(_bench_dump(tmp_path, 1, "--impl", "reference")[1], depth)


@pytest.mark.gpu
def test_product_arm_dumps_the_last_timed_bfs(tmp_path):
    import numpy as np
    import oracle
    from essentials_b200 import graphgen as gg
    d, depth, src = _bench_dump(tmp_path, 0, "--no-extras", "--no-cpu", "--no-e2e")
    assert d["steps"] == 3 and d["parity_ok"] is True
    off, col, _ = gg.rmat_csr(12, 16).host()
    assert np.array_equal(depth, oracle.bfs(off, col, src).astype(np.float64))


def test_dump_of_a_long_output_is_a_fixed_sample(tmp_path):
    """Above DUMP_SAMPLE entries (every scale-26 run): DUMP_SAMPLE values at fixed positions, listed beside them."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    n = bench.DUMP_SAMPLE * 3 + 5
    depth = torch.randint(0, 2**31 - 1, (n,), dtype=torch.int32)
    for run in (0, 1):
        bench.dump_outputs(str(tmp_path / f"d{run}"), {"bfs_depth": depth})
    vals, idx = (np.load(str(tmp_path / "d0" / f)) for f in ("bfs_depth.npy", "bfs_depth_index.npy"))
    assert vals.dtype == idx.dtype == np.float64 and vals.size == idx.size == bench.DUMP_SAMPLE
    assert vals.nbytes + idx.nbytes <= 64 * 2**20
    assert np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < n
    assert np.array_equal(vals, depth.numpy()[idx.astype(np.int64)].astype(np.float64))
    for f in ("bfs_depth.npy", "bfs_depth_index.npy"):
        assert np.array_equal(np.load(str(tmp_path / "d1" / f)), np.load(str(tmp_path / "d0" / f)))


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--scale", "10",
                          "--steps", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and not out.stdout.strip()


def test_default_workload_is_the_north_star():
    """No flags = Kronecker scale-26 (BASELINE.json north_star) at every N: strong scaling."""
    sys.path.insert(0, ROOT)
    import bench
    old = sys.argv
    try:
        sys.argv = ["bench.py"]
        args = bench.parse()
    finally:
        sys.argv = old
    assert args.scale == 0 and bench.NORTH_STAR_SCALE == 26 and not args.weak


def test_certificates_accept_the_oracle_and_reject_corruption():
    """bench.py's full-size parity checks: the BFS / SSSP certificates pass on the oracle's answers (whole graph and
    a 2-way row partition) and flag any single corrupted entry."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    import oracle
    from essentials_b200 import graphgen as gg
    csr = gg.rmat_csr(11, 8, weights="hash", device="cpu")
    off, col, val = csr.host()
    src = gg.pick_sources(csr, 1)[0]
    depth = torch.from_numpy(oracle.bfs(off, col, src))
    dist = torch.from_numpy(oracle.sssp(off, col, val, src))
    assert bench.bfs_certificate(csr.offsets, csr.indices, depth, src) == 0
    assert bench.sssp_certificate(csr.offsets, csr.indices, csr.values, dist, src) == 0
    half = csr.n // 2
    for lo, hi in ((0, half), (half, csr.n)):  # a rank's rows against the full result array
        part = gg.rmat_csr(11, 8, weights="hash", device="cpu", row_range=(lo, hi))
        assert bench.bfs_certificate(part.offsets, part.indices, depth, src, row_begin=lo) == 0
        assert bench.sssp_certificate(part.offsets, part.indices, part.values, dist, src, row_begin=lo) == 0
    reached = (depth != bench.INF).nonzero().flatten()
    v = int(reached[reached != src][7])
    for delta in (1, -1):
        bad = depth.clone()
        bad[v] += delta
        assert bench.bfs_certificate(csr.offsets, csr.indices, bad, src) > 0
    bad = depth.clone()
    bad[v] = bench.INF  # a reached vertex reported unreached
    assert bench.bfs_certificate(csr.offsets, csr.indices, bad, src) > 0
    for factor in (0.5, 1.5):
        badd = dist.clone()
        badd[v] *= factor
        assert bench.sssp_certificate(csr.offsets, csr.indices, csr.values, badd, src) > 0


def test_product_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return  # on a GPU box the product arm is exercised by the driver itself
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0",
                          "--scale", "10"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and not out.stdout.strip(), "no CPU fallback: nothing may be printed as a result"
