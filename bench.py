#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on its north-star config: BFS GTEPS on a Kronecker scale-26 edge-factor-16 graph.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A step is one BFS (one pass of the frontier-operator hot path) from one pseudo-random non-isolated source of the
synthetic graph; the K timed steps use K different sources. GTEPS = directed edges leaving reached vertices (m',
SURVEY.md §8d) summed over the steps / time. Rank 0 prints ONE JSON line.

  value        graph resident in HBM, K x ess_bfs (problem reset + enact), CUDA events on the library's stream, max
               over ranks. N > 1 without --scale = STRONG scaling of the same scale-26 graph (1-D vertex partition).
  parity       every timed source is checked on the device by the BFS certificate (bfs_certificate below: d[s] = 0,
               no edge spans more than one level or joins reached to unreached, every reached vertex has a parent one
               level up — together these PROVE d is the BFS depth array); one source is also compared with the
               reference's own bfs_cpu; at N > 1 every rank certifies its rows against the all-gathered depths (and
               at N = 2 they are also compared with a single-GPU ess_bfs on rank 0). A mismatch sets parity_ok false
               and the exit code to 3.
  e2e          the same K sources through the public host API with HOST buffers: every step hands the CSR arrays in
               pinned host memory to ess_graph_create_from_host (H2D copy + graph handle incl. the bottom-up hints,
               built under the copy), runs BFS, copies the depth array back and destroys the handle.
  roofline     dominant kernel class of an instrumented repeat of the K steps (CUDA events around every launch):
               algorithmic bytes / kernel time vs the measured HBM peak in MEASURED_PEAKS.json (DESIGN.md §5).
  cpu_baseline the reference's own bfs_cpu (oracle/_ref, 1 thread) on one source of the same graph, rank 0, N=1.
  sssp / other_configs   BASELINE configs 2-5 side runs (SSSP lines carry their own roofline block).
  --impl reference   times the reference's CPU implementation alone on the SAME graph and sources, one bfs_cpu per
               host thread (the only other place oracle/ is executed).
  --dump-outputs DIR   after the timed steps, writes the depth array of the last timed BFS (what ess_bfs hands its
               caller) to DIR/bfs_depth.npy, float64; above DUMP_SAMPLE vertices a fixed strided sample of positions,
               listed in DIR/bfs_depth_index.npy. Graph and sources are seeded, so two builds run with the same
               arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

INF = 2**31 - 1
FLT_MAX = 3.4028234663852886e38
NORTH_STAR_SCALE = 26
T0 = time.time()


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scale", type=int, default=0,
                    help="Kronecker scale of the headline workload; default 26 (BASELINE north star) at every N, i.e. "
                         "strong scaling; --weak runs 2^24*16 generated edges per GPU instead (scale 24 + log2 N)")
    ap.add_argument("--weak", action="store_true")
    ap.add_argument("--edge-factor", type=int, default=16)
    ap.add_argument("--lb", default="merge_path")
    ap.add_argument("--direction", default="optimized")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--nccl-exchange", action="store_true",
                    help="multi-GPU: NCCL send/recv + all_gather instead of the peer-memory exchange kernels")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the side runs (configs 2-5, reference GPU)")
    ap.add_argument("--extras-budget-s", type=float, default=420.0,
                    help="side runs are skipped once the process has been running this long")
    ap.add_argument("--cpu-threads", type=int, default=0, help="reference arm: concurrent bfs_cpu runs (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output of the last timed step as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_SAMPLE = 1 << 21  # entries kept per dumped output: 16 MiB of float64 values plus 16 MiB of positions


def dump_outputs(out_dir, arrays):
    """Writes each named tensor as out_dir/<name>.npy in float64 (exact for int32 depths and float32 distances). A
    tensor longer than DUMP_SAMPLE keeps DUMP_SAMPLE positions at a fixed stride, the same for every run and every
    install (graphgen permutes vertex ids, so a stride samples the graph evenly); the positions go to
    out_dir/<name>_index.npy."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        n = t.numel()
        if n > DUMP_SAMPLE:
            idx = torch.arange(DUMP_SAMPLE, dtype=torch.int64) * (n // DUMP_SAMPLE)
            vals = t[idx.to(t.device)]
            np.save(os.path.join(out_dir, f"{name}_index.npy"), idx.numpy().astype(np.float64))
        else:
            vals = t
        np.save(os.path.join(out_dir, f"{name}.npy"), vals.cpu().numpy().astype(np.float64))


def check_sources(srcs, count):
    """The timed loop runs one step per source: fewer sources than asked for would silently shorten it."""
    if len(srcs) != count:
        raise SystemExit(f"bench.py: the graph has only {len(srcs)} usable sources, {count} needed "
                         f"(--steps + --warmup)")


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel_class):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    `ncu --set full` capture (profiles/ncu_traffic.json says which capture); None when there is none."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f).get(kernel_class, {}).get("bytes_per_launch")
    except Exception:
        return None


def workload_config(scale, edge_factor, n, m, steps):
    """The workload description both arms print (the driver compares the two `config` objects)."""
    return {"workload": f"BFS kron scale-{scale} ef-{edge_factor} symmetrised, {steps} random non-isolated sources",
            "scale": scale, "edge_factor": edge_factor, "n": int(n), "m": int(m),
            "teps_edges": "directed edges leaving reached vertices (m')",
            "l2": "CSR (%.2f GB) exceeds the 126 MB L2; no flush between steps" % ((m * 4 + n * 4) / 1e9)}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i] == "Active"})
        mx = max((int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()), default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons,
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------- result certificates
def _row_chunks(offsets, max_edges=1 << 27):
    """Row ranges [r0, r1) of a CSR whose edge counts stay below max_edges (bounds the temporaries below)."""
    import torch
    n = offsets.numel() - 1
    total = int(offsets[-1].item()) - int(offsets[0].item())
    parts = max(1, (total + max_edges - 1) // max_edges)
    targets = torch.arange(1, parts, device=offsets.device, dtype=torch.int64) * (total // parts) + int(offsets[0].item())
    cuts = torch.searchsorted(offsets.to(torch.int64), targets).tolist() if parts > 1 else []
    bounds = [0] + [min(max(int(c), 0), n) for c in cuts] + [n]
    return [(bounds[i], bounds[i + 1]) for i in range(len(bounds) - 1) if bounds[i + 1] > bounds[i]]


def bfs_certificate(offsets, indices, depth, source, row_begin=0):
    """Number of violations of the three conditions that characterise BFS depths (0 = `depth` IS the depth array):
      (a) depth[source] == 0;
      (b) every edge joins two reached or two unreached vertices, and reached endpoints differ by at most 1;
      (c) every reached vertex other than the source has a neighbour exactly one level up.
    (c) gives depth >= distance (follow parents down to the source), (b) gives depth <= distance (depth grows by at
    most 1 along a shortest path), so all three together prove equality. Pure torch on the device that holds the
    arrays; `offsets`/`indices` may be a row range of a partition (global column ids, rows row_begin ...), `depth`
    is the full array. Size independent: this is the parity check at BASELINE's full sizes."""
    import torch
    bad = 0 if int(depth[source].item()) == 0 else 1
    base = int(offsets[0].item())
    for r0, r1 in _row_chunks(offsets):
        e0, e1 = int(offsets[r0].item()) - base, int(offsets[r1].item()) - base
        deg = (offsets[r0 + 1:r1 + 1] - offsets[r0:r1]).to(torch.int64)
        d_row = depth[row_begin + r0:row_begin + r1]
        if e1 > e0:
            rows = torch.repeat_interleave(torch.arange(r1 - r0, device=depth.device, dtype=torch.int32), deg)
            d_u = d_row[rows.long()]
            d_v = depth[indices[e0:e1].long()]
            reach_u, reach_v = d_u != INF, d_v != INF
            bad += int((reach_u != reach_v).sum().item())
            both = reach_u & reach_v
            bad += int(((d_u - d_v).abs()[both] > 1).sum().item())
            best = torch.full((r1 - r0,), INF, dtype=torch.int32, device=depth.device)
            best.scatter_reduce_(0, rows.long(), d_v, "amin", include_self=True)
            del rows, d_u, d_v, reach_u, reach_v, both
        else:
            best = torch.full((r1 - r0,), INF, dtype=torch.int32, device=depth.device)
        need = (d_row != INF) & (d_row != 0)
        bad += int((best[need] != d_row[need] - 1).sum().item())
        zeros = (d_row == 0).nonzero().flatten() + row_begin + r0  # only the source may sit at level 0
        bad += int((zeros != source).sum().item())
    return bad


def sssp_certificate(offsets, indices, values, dist, source, row_begin=0):
    """Violations of the fixed-point conditions of single-source shortest paths in float arithmetic: dist[source] == 0;
    no edge can still relax (dist[v] <= fl(dist[u] + w)); every reached vertex but the source has a tight in-edge
    (dist[v] == fl(dist[u] + w) for some neighbour u; the graphs here are symmetric, so rows list in-neighbours)."""
    import torch
    bad = 0 if float(dist[source].item()) == 0.0 else 1
    base = int(offsets[0].item())
    for r0, r1 in _row_chunks(offsets):
        e0, e1 = int(offsets[r0].item()) - base, int(offsets[r1].item()) - base
        deg = (offsets[r0 + 1:r1 + 1] - offsets[r0:r1]).to(torch.int64)
        d_row = dist[row_begin + r0:row_begin + r1]
        best = torch.full((r1 - r0,), FLT_MAX, dtype=torch.float32, device=dist.device)
        if e1 > e0:
            rows = torch.repeat_interleave(torch.arange(r1 - r0, device=dist.device, dtype=torch.int32), deg).long()
            d_nbr = dist[indices[e0:e1].long()]
            via = torch.where(d_nbr < FLT_MAX, d_nbr + values[e0:e1], torch.full_like(d_nbr, FLT_MAX))
            bad += int((via < d_row[rows]).sum().item())  # a relaxable edge
            best.scatter_reduce_(0, rows, via, "amin", include_self=True)
            del rows, d_nbr, via
        need = d_row < FLT_MAX
        if row_begin + r0 <= source < row_begin + r1:
            need[source - row_begin - r0] = False
        bad += int((best[need] != d_row[need]).sum().item())
    return bad


def reached_work(csr, depth):
    """(n', m') of a depth array: reached vertices and the directed edges leaving them."""
    import torch
    r = depth != INF
    return int(r.sum()), int(csr.degrees().to(torch.int64)[r].sum())


# --------------------------------------------------------------------------------------------- reference arm
def run_reference(args, rank, world):
    """The reference's own CPU BFS (examples/algorithms/bfs/bfs_cpu.hxx via oracle/_ref, or our port when the
    reference did not compile) on the SAME graph and sources as our arm; one single-threaded bfs_cpu per host thread."""
    if rank != 0:
        return
    from concurrent.futures import ThreadPoolExecutor

    import numpy as np
    import torch

    import oracle
    from essentials_b200 import graphgen as gg
    K, W = args.steps, max(args.warmup, 0)
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    csr = gg.rmat_csr(args.scale, args.edge_factor, device=dev)
    srcs = gg.pick_sources(csr, K + W)
    check_sources(srcs, K + W)
    n, m = csr.n, csr.m
    off = csr.offsets.cpu().numpy()
    col = csr.indices.cpu().numpy()
    del csr
    if dev == "cuda":
        torch.cuda.empty_cache()
    deg = np.diff(off.astype(np.int64))
    use_ref = oracle.have_ref() and off.dtype.itemsize == 4
    kind = "reference" if use_ref else "port"
    if use_ref:
        G = oracle.RefGraph(off, col)
        one = G.bfs
    else:
        def one(s):
            return oracle.bfs(off, col, s, return_ms=True)
    # concurrency: one source per host thread, bounded by memory (every bfs_cpu call copies the CSR, bfs_cpu.hxx:25-27)
    threads = args.cpu_threads or (os.cpu_count() or 1)
    try:
        import psutil
        per_run = off.nbytes + col.nbytes + 48 * n + (1 << 28)  # bfs_cpu's private CSR copy + dist + pred + queue
        threads = max(1, min(threads, int(psutil.virtual_memory().available * 0.7 // per_run)))
    except Exception:
        threads = min(threads, 8)
    threads = max(1, min(threads, K))

    def work(s):
        d, ms = one(s)
        return int(deg[d != INF].sum()), float(ms)

    with ThreadPoolExecutor(threads) as pool:
        list(pool.map(work, srcs[:W]))
        t0 = time.time()
        res = list(pool.map(work, srcs[W:]))
        wall = time.time() - t0
    if args.dump_outputs:  # work() keeps no depth arrays (K of them would not fit at scale 26): rerun the last source
        dump_outputs(args.dump_outputs, {"bfs_depth": torch.from_numpy(one(srcs[-1])[0])})
    edges = sum(r[0] for r in res)
    search_ms = sum(r[1] for r in res)
    val = edges / wall / 1e9
    sample = (f"{K} full BFS runs of the reference's single-threaded bfs_cpu on the workload graph itself, {threads} "
              f"at a time on {threads} host threads (of {os.cpu_count()}); wall {wall:.1f} s for the {K} timed runs "
              f"(search loops alone: {search_ms / 1e3:.1f} thread-seconds = {edges / max(search_ms, 1e-9) / 1e6:.3f} "
              f"GTEPS per thread, as bfs_cpu.hxx:35,65-67 times itself)")
    line = {
        "impl": "reference", "metric": "BFS GTEPS", "value": val, "unit": "GTEPS", "n_gpus": args.gpus,
        "steps": K, "warmup": W, "ms_per_step": wall * 1e3 / K, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": workload_config(args.scale, args.edge_factor, n, m, K),
        "cpu_baseline": {"value": val, "unit": "GTEPS", "cores": threads, "kind": kind, "sample": sample,
                         "per_thread_gteps": edges / max(search_ms, 1e-9) / 1e6},
        "e2e": {"value": val, "unit": "GTEPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- our arm, one GPU
def bfs_roofline(prof, acc, n, sE, K, ms, edges, verts, peak_gbs, peak_src):
    """Roofline block of the dominant BFS kernel class. Byte model (DESIGN.md §5) — what the kernels must move:
    bottom-up: 3 bitmaps per level + 8 B per probed hint (head id + frontier word) + 8 B per in-edge walked
    (column id + frontier word) + the row bounds of every vertex whose hint missed + 4 B per adopted vertex (depth);
    top-down: SURVEY §8d's 8 B per expanded edge (column id + visited word) + (2 sE + 12) B per expanded vertex."""
    bytes_by_class = {
        "pull_step": acc["pull_steps"] * 3 * (n / 8) + acc["pull_vertices"] * 8 + acc["pull_edges"] * 8
                     + acc["pull_misses"] * 2 * sE + acc["pull_found"] * 4,
        "push_expand": acc["push_edges"] * 8 + acc["push_vertices"] * (2 * sE + 12),
    }
    kernel_ms = {k: v[0] for k, v in prof.items()}
    dom = max(bytes_by_class, key=lambda k: kernel_ms.get(k, 0.0))
    d_ms, d_launches = prof[dom]
    achieved = bytes_by_class[dom] / (d_ms * 1e-3) / 1e9 if d_ms > 0 else 0.0
    graph500_bytes = 8 * edges + (2 * sE + 12) * verts
    return {
        "bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
        "frac": achieved / peak_gbs, "traffic": ncu_traffic(dom), "peak_source": peak_src,
        "frac_of_nominal_8000_gbs": achieved / 8000.0,
        "launches": d_launches, "avg_launch_ms": d_ms / max(d_launches, 1),
        "algorithmic_bytes_per_launch": bytes_by_class[dom] / max(d_launches, 1),
        "kernel_ms_per_step": {k: v / K for k, v in kernel_ms.items() if v},
        "kernel_share_of_step": sum(kernel_ms.values()) / ms if ms else None,
        "share_of_step": d_ms / ms if ms else None,
        "work_per_step": {k: v / K for k, v in acc.items()},
        "whole_bfs_effective_gbs": graph500_bytes / (ms * 1e-3) / 1e9,
        "secondary_ceiling": {
            "what": "L1TEX wavefronts of divergent 4-byte gathers (frontier/visited word probes, depth and row-bound "
                    "reads): one 128-byte line per lane at ~2.07 cycles per line per SM (B300_MICROARCH.md, LDG "
                    "model) = 148 x 1.965 GHz / 2.07 = 140.5 G gathers/s; ncu evidence in profiles/",
            "gathers_per_s_ceiling": 148 * 1.965e9 / 2.07,
        },
        "note": "achieved counts bytes the kernel has to move (edges skipped by direction optimisation are not "
                "counted); whole_bfs_effective_gbs applies SURVEY §8d's 8*m'+(2*sE+12)*n' to the TEPS-counted edges "
                "and can exceed the peak for exactly that reason — it is work skipped, not data moved",
    }


def run_single(args, rank, local_rank):
    import numpy as np
    import torch

    import essentials_b200 as ess
    from essentials_b200 import graphgen as gg

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.Stream(device=dev)
    peak_gbs, peak_src = peaks()
    K, W = args.steps, max(args.warmup, 0)
    with torch.cuda.stream(stream):
        csr = gg.rmat_csr(args.scale, args.edge_factor, device=dev)
        ctx = ess.Context(local_rank, stream=stream)
        graph = ess.Graph(csr)
        depth = torch.empty(csr.n, dtype=torch.int32, device=dev)
    stream.synchronize()
    n, m, offset_bits = csr.n, csr.m, graph.offset_bits
    srcs = gg.pick_sources(csr, K + W)
    check_sources(srcs, K + W)
    timed = srcs[W:]

    def one_bfs(s, g=None):
        return ess.bfs(ctx, g or graph, s, lb=args.lb, direction=args.direction, out=depth)[1]

    # ---- untimed pre-pass: per-source work (n', m') and the certificate of every timed source --------------
    work, violations = {}, 0
    with torch.cuda.stream(stream):
        for s in srcs:
            one_bfs(s)
            work[s] = reached_work(csr, depth)
            if s in timed:
                violations += bfs_certificate(csr.offsets, csr.indices, depth, s)
        for s in srcs[:W]:  # warm-up proper (allocator pools, clocks)
            one_bfs(s)
    stream.synchronize()
    edges = sum(work[s][1] for s in timed)
    verts = sum(work[s][0] for s in timed)

    # ---- timed region: K steps, device events on the launching stream, sync on both sides -------------------
    launches0 = ctx.launches()
    sampler = ClockSampler(local_rank)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    enact_ms = 0.0
    with torch.cuda.stream(stream):
        e0.record(stream)
        for s in timed:
            enact_ms += one_bfs(s)["enact_ms"]
        e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    launches = ctx.launches() - launches0
    value = edges / (ms * 1e-3) / 1e9
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"bfs_depth": depth})  # depth still holds the last timed source's BFS

    out = {
        "metric": "BFS GTEPS", "value": value, "unit": "GTEPS", "n_gpus": 1, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "int32", "data": "synthetic",
        "config": workload_config(args.scale, args.edge_factor, n, m, K),
        "implementation": {"advance": f"{args.lb}/{args.direction}", "edge_t_bits": offset_bits,
                           "parallelism": "single-gpu"},
        "enact_ms_per_step": enact_ms / K,
        "gpu_launches": launches,
        "clocks": clocks,
        "parity": {"certificate_violations": violations, "sources_certified": len(timed),
                   "what": "BFS certificate (bench.py:bfs_certificate) of every timed source on the full graph"},
    }
    parity_ok = violations == 0

    # ---- roofline: instrumented repeat of the same K steps -------------------------------------------------
    sE = offset_bits // 8
    acc = {k: 0 for k in ("pull_vertices", "pull_edges", "push_vertices", "push_edges", "pull_steps", "pull_misses",
                          "pull_found", "push_found")}
    with torch.cuda.stream(stream):
        ctx.profile(True)
        for s in timed:
            info = one_bfs(s)
            for k in acc:
                acc[k] += info[k]
        prof = ctx.profile_read()
        ctx.profile(False)
    out["roofline"] = bfs_roofline(prof, acc, n, sE, K, ms, edges, verts, peak_gbs, peak_src)

    # ---- e2e: host buffers in, host buffer out, graph handle (incl. hints) rebuilt, every step -------------
    last_depth = None
    if not args.no_e2e:
        h_csr = csr.pinned()  # the caller's graph: host arrays in page-locked memory
        h_depth = torch.empty(n, dtype=torch.int32).pin_memory()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):
            ess.Graph.from_host(ctx, h_csr).close()  # untimed: the device blocks of the handle come from the driver once
            torch.cuda.synchronize()
            f0.record(stream)
            for s in timed:
                # ess_graph_create_from_host: H2D of offsets + indices into device arrays the handle owns, graph views,
                # bottom-up hints and isolated-vertex bitmap (built chunk by chunk under the copy)
                g = ess.Graph.from_host(ctx, h_csr)
                one_bfs(s, g)
                h_depth.copy_(depth, non_blocking=True)
                stream.synchronize()
                g.close()
            f1.record(stream)
        torch.cuda.synchronize()
        ems = f0.elapsed_time(f1)
        out["e2e"] = {"value": edges / (ems * 1e-3) / 1e9, "unit": "GTEPS",
                      "h2d_bytes_per_step": int(h_csr.nbytes()),
                      "d2h_bytes_per_step": int(n * 4), "ms_per_step": ems / K,
                      "what": "per step, from host arrays: ess_graph_create_from_host (CSR offsets+indices H2D from "
                              "pinned memory in chunks, graph views, bottom-up hints and isolated-vertex bitmap built "
                              "under the copy; nothing is reused between steps), ess_bfs, depth D2H, "
                              "ess_graph_destroy"}
        last_depth = h_depth.numpy().copy()
        del h_csr
        with torch.cuda.stream(stream):  # the host-array path must give the depths of the resident graph
            one_bfs(timed[-1])
        stream.synchronize()
        out["e2e"]["depths_equal_resident_graph"] = bool(torch.equal(depth.cpu(), h_depth))
        parity_ok = parity_ok and out["e2e"]["depths_equal_resident_graph"]

    # ---- CPU baseline: the reference's bfs_cpu, one source of the same graph --------------------------------
    if not args.no_cpu:
        import oracle
        s = timed[-1]
        if last_depth is None:
            with torch.cuda.stream(stream):
                one_bfs(s)
            stream.synchronize()
            last_depth = depth.cpu().numpy()
        off = csr.offsets.cpu().numpy()
        col = csr.indices.cpu().numpy()
        if oracle.have_ref() and off.dtype.itemsize == 4:
            G = oracle.RefGraph(off, col)
            d_cpu, cpu_ms = G.bfs(s)
            G.close()
            kind = "reference"
        else:
            d_cpu, cpu_ms = oracle.bfs(off, col, s, return_ms=True)
            kind = "port"
        same = bool(np.array_equal(d_cpu, last_depth))
        out["cpu_baseline"] = {
            "value": work[s][1] / (cpu_ms * 1e-3) / 1e9, "unit": "GTEPS", "cores": 1, "kind": kind,
            "sample": f"1 BFS (source {s}) on the full workload graph, search time only ({cpu_ms / 1e3:.1f} s)",
            "depths_equal_gpu": same}
        parity_ok = parity_ok and same
        del off, col, d_cpu
    out["parity_ok"] = parity_ok

    # ---- side measurements (BASELINE configs 2-4 and the reference's own GPU path); never fatal -------------
    if not args.no_extras:
        try:
            del csr, graph, depth
            torch.cuda.empty_cache()
            side_runs(args, ctx, dev, out, peak_gbs)
        except Exception as e:  # the headline line must survive anything here
            out.setdefault("other_configs", {})["error"] = repr(e)[:300]
    print(json.dumps(out), flush=True)
    return 0 if out["parity_ok"] else 3


def sssp_roofline(n_reached, m_reached, sE, ms, peak_gbs):
    """SURVEY §8d: B = m'(sV + sW + sW) + n'(2 sE + 3 sV + sW), every edge counted once (Dijkstra work)."""
    b = m_reached * 12 + n_reached * (2 * sE + 16)
    gbs = b / (ms * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": gbs, "peak": peak_gbs, "unit": "GB/s", "frac": gbs / peak_gbs,
            "algorithmic_bytes": b}


def side_runs(args, ctx, dev, out, peak_gbs):
    """BASELINE configs 2, 3, 4 and the reference's own GPU implementation on this same device."""
    import torch

    import essentials_b200 as ess
    import oracle
    from essentials_b200 import graphgen as gg
    res = out.setdefault("other_configs", {})

    def over_budget(name):
        if time.time() - T0 > args.extras_budget_s:
            res[name] = {"skipped": f"time budget ({args.extras_budget_s:.0f} s since start)"}
            return True
        return False

    # ---- config 2: BFS on Kronecker scale-24, block_mapped vs merge_path, with and without the push/pull switch,
    #      every source compared with the reference's own GPU BFS (block_mapped + Thrust, built for sm_100)
    if not over_budget("bfs_kron24"):
        csr = gg.rmat_csr(24, args.edge_factor, device=dev)
        g = ess.Graph(csr)
        srcs = gg.pick_sources(csr, 8)
        deg = csr.degrees().to(torch.int64)
        rows = {}
        ref_depths, ref_ms = {}, []
        have_ref_gpu = oracle.have_ref_gpu() and csr.offsets.dtype == torch.int32
        if have_ref_gpu:
            oracle.ref_gpu_run("bfs", csr, srcs[0])  # warm
            for s in srcs:
                d, t = oracle.ref_gpu_run("bfs", csr, s)
                ref_depths[s] = d
                ref_ms.append(t)
        m_r = {}
        for lb in ("block_mapped", "merge_path"):
            for direction in ("forward", "optimized"):
                ess.bfs(ctx, g, srcs[0], lb=lb, direction=direction)  # warm
                t_ms, equal = [], True
                for s in srcs:
                    d, info = ess.bfs(ctx, g, s, lb=lb, direction=direction)
                    t_ms.append(info["enact_ms"])
                    m_r[s] = int(deg[d != INF].sum())
                    if have_ref_gpu:
                        equal = equal and bool(torch.equal(d, ref_depths[s]))
                tot_e = sum(m_r[s] for s in srcs)
                rows[f"{lb}/{direction}"] = {"enact_ms_mean": sum(t_ms) / len(t_ms), "gteps": tot_e / sum(t_ms) / 1e6,
                                             "bytes_8_per_edge_gbs": 8 * tot_e / sum(t_ms) / 1e6,
                                             "depths_equal_reference_gpu": equal if have_ref_gpu else None}
                if have_ref_gpu and not equal:
                    out["parity_ok"] = False
        res["bfs_kron24"] = {"n": csr.n, "m": csr.m, "sources": len(srcs), "ours": rows}
        if have_ref_gpu:
            tot_e = sum(m_r[s] for s in srcs)
            res["bfs_kron24"]["reference_gpu"] = {"enact_ms_mean": sum(ref_ms) / len(ref_ms),
                                                 "gteps": tot_e / sum(ref_ms) / 1e6}
        ref_depths.clear()
        # ---- SSSP on the same graph (weights from the symmetric pair hash): dense delta vs the frontier recipe
        if not over_budget("sssp_kron24"):
            from dataclasses import replace
            r = torch.repeat_interleave(torch.arange(csr.n, device=dev, dtype=torch.int64), deg)
            weighted = replace(csr, values=gg.pair_weights(r, csr.indices.to(torch.int64)))
            del r
            wg = ess.Graph(weighted)
            runs, viol = [], 0
            for s in srcs[:3]:
                for _ in range(2):  # second run: buffers warm
                    d_delta, i_delta = ess.sssp_delta(ctx, wg, s)
                    d_front, i_front = ess.sssp(ctx, wg, s, lb="merge_path")
                reached = d_delta < FLT_MAX
                n_r, me = int(reached.sum()), int(deg[reached].sum())
                viol += sssp_certificate(weighted.offsets, weighted.indices, weighted.values, d_delta, s)
                runs.append({"source": s, "delta_enact_ms": i_delta["enact_ms"], "delta_rounds": i_delta["rounds"],
                             "delta_gteps": me / i_delta["enact_ms"] / 1e6,
                             "frontier_merge_path_enact_ms": i_front["enact_ms"],
                             "roofline": sssp_roofline(n_r, me, 4, i_delta["enact_ms"], peak_gbs),
                             "distances_equal": bool(torch.equal(d_delta, d_front))})
            res["sssp_kron24"] = {"weights": "uniform [1,64) dyadic, symmetric hash", "runs": runs,
                                  "certificate_violations": viol}
            if viol or not all(r["distances_equal"] for r in runs):
                out["parity_ok"] = False
            del wg, weighted, d_delta, d_front
        del g, csr, deg
        torch.cuda.empty_cache()
    # ---- config 3: SSSP on the 4900 x 4900 grid
    if not over_budget("sssp_grid_4900"):
        grid = gg.grid_csr(4900, 4900, device=dev)
        gg_graph = ess.Graph(grid)
        ess.sssp_near_far(ctx, gg_graph, 0)  # warm
        d_nf, i_nf = ess.sssp_near_far(ctx, gg_graph, 0)
        d_lc, i_lc = ess.sssp(ctx, gg_graph, 0, lb="block_mapped")
        viol = sssp_certificate(grid.offsets, grid.indices, grid.values, d_nf, 0)
        res["sssp_grid_4900"] = {"n": grid.n, "m": grid.m, "near_far_enact_ms": i_nf["enact_ms"],
                                 "near_far_gteps": grid.m / i_nf["enact_ms"] / 1e6, "near_far_levels": i_nf["levels"],
                                 "us_per_level": 1e3 * i_nf["enact_ms"] / max(i_nf["levels"], 1),
                                 "relaxations_per_edge": i_nf["relaxations"] / grid.m,
                                 "label_correcting_block_mapped_enact_ms": i_lc["enact_ms"],
                                 "roofline": sssp_roofline(grid.n, grid.m, 4, i_nf["enact_ms"], peak_gbs),
                                 "certificate_violations": viol,
                                 "distances_equal": bool(torch.equal(d_nf, d_lc))}
        if viol or not res["sssp_grid_4900"]["distances_equal"]:
            out["parity_ok"] = False
        if oracle.have_ref_gpu():
            ref_dist, ref_ms = oracle.ref_gpu_run("sssp", grid, 0)
            res["sssp_grid_4900"].update(reference_gpu_enact_ms=ref_ms,
                                         equal_reference_gpu=bool(torch.equal(d_nf, ref_dist)))
            del ref_dist
        del gg_graph, grid, d_nf, d_lc
        torch.cuda.empty_cache()
    # ---- config 4: PageRank on directed RMAT scale-25
    if not over_budget("pagerank_rmat25"):
        pr_csr = gg.rmat_csr(25, args.edge_factor, symmetric=False, weights="ones", device=dev)
        pr_graph = ess.Graph(pr_csr, csc=ess.transpose(pr_csr))
        p_pull, i_pull = ess.pagerank(ctx, pr_graph, pull=True)
        p_push, i_push = ess.pagerank(ctx, pr_graph, lb="merge_path", pull=False)
        rel = ((p_pull.double() - p_push.double()).abs().sum() / p_pull.double().sum()).item()
        it = max(i_pull["iterations"], 1)
        per_iter_bytes = pr_csr.m * 12 + pr_csr.n * (2 * 4 + 9 * 4)  # SURVEY §8d
        res["pagerank_rmat25"] = {"n": pr_csr.n, "m": pr_csr.m, "iterations": i_pull["iterations"],
                                  "pull_ms_per_iteration": i_pull["enact_ms"] / it,
                                  "push_merge_path_ms_per_iteration": i_push["enact_ms"] / max(i_push["iterations"], 1),
                                  "pull_gteps": pr_csr.m * it / i_pull["enact_ms"] / 1e6,
                                  "roofline": {"bound": "hbm", "achieved": per_iter_bytes * it / i_pull["enact_ms"] / 1e6,
                                               "peak": peak_gbs, "unit": "GB/s",
                                               "frac": per_iter_bytes * it / i_pull["enact_ms"] / 1e6 / peak_gbs},
                                  "rel_l1_push_vs_pull": rel}
        if oracle.have_ref_gpu():
            ref_p, ref_ms = oracle.ref_gpu_run("pr", pr_csr, 0.85, 1e-6)
            res["pagerank_rmat25"].update(reference_gpu_enact_ms=ref_ms, ours_pull_enact_ms=i_pull["enact_ms"],
                                          rel_l1_vs_reference_gpu=((p_pull.double() - ref_p.double()).abs().sum()
                                                                   / ref_p.double().sum()).item())


# --------------------------------------------------------------------------------------------- our arm, N GPUs
def run_distributed(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist

    import essentials_b200 as ess
    from essentials_b200 import dist as edist
    from essentials_b200 import graphgen as gg

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.Stream(device=dev)
    peak_gbs, peak_src = peaks()
    K, W = args.steps, max(args.warmup, 0)
    if args.nccl_exchange:
        ess.tune("dist_peer_exchange", 0)

    def all_max(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_sum(x):
        t = torch.tensor([x], device=dev, dtype=torch.int64)
        dist.all_reduce(t)
        return int(t.item())

    def measure(scale, steps, warm, sssp_steps=0, check_single=False, dump_dir=None):
        """One partitioned workload: timed BFS (and SSSP) steps + certificates. Returns a dict (same on every rank)."""
        runner = edist.build_partitioned(scale, args.edge_factor, rank, world, dev, stream,
                                         weights="hash" if sssp_steps else "none")
        stream.synchronize()
        with torch.cuda.stream(stream):
            srcs = runner.pick_sources(steps + warm)
        check_sources(srcs, steps + warm)
        timed = srcs[warm:]
        work, viol = {}, 0
        with torch.cuda.stream(stream):
            for s in srcs:
                runner.bfs(s)
                work[s] = runner.reached_work()
                if s in timed:
                    full = runner.gather_depth()
                    viol += bfs_certificate(runner.csr.offsets, runner.csr.indices, full, s, runner.row_begin)
                    del full
            for s in srcs[:warm]:
                runner.bfs(s)
        stream.synchronize()
        viol = all_sum(viol)
        edges = sum(work[s][1] for s in timed)
        launches0 = runner.backend.launches()
        sampler = ClockSampler(local_rank) if rank == 0 else None
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for s in timed:
                runner.bfs(s)
            e1.record(stream)
        torch.cuda.synchronize()
        dist.barrier()
        ms = all_max(e0.elapsed_time(e1))
        if dump_dir:
            with torch.cuda.stream(stream):
                full = runner.gather_depth()  # collective: the last timed source's depths, all partitions
            stream.synchronize()
            if rank == 0:
                dump_outputs(dump_dir, {"bfs_depth": full})
            del full
        r = {"scale": scale, "n": runner.n_global, "m": runner.m_global, "offset_bits": runner.offset_bits,
             "steps": steps, "ms": ms, "edges": edges, "gteps": edges / (ms * 1e-3) / 1e9,
             "certificate_violations": viol, "launches": runner.backend.launches() - launches0,
             "clocks": sampler.stop() if sampler else None, "levels": runner.levels,
             "pull_levels": runner.pull_levels, "nvlink_bytes": runner.bytes_exchanged,
             "exchange_kind": runner.exchange_kind()}
        if check_single and scale <= 26 and world <= 2:
            # (N <= 2: the configuration this cross-check was validated on; at every N the certificate above proves the
            # depths) rank 0 rebuilds the whole graph and runs the single-GPU ess_bfs on the same sources
            equal, failure = True, None
            fulls = []
            with torch.cuda.stream(stream):
                for s in timed[:4]:
                    runner.bfs(s)
                    full = runner.gather_depth()
                    if rank == 0:
                        fulls.append(full)
                    del full
            stream.synchronize()
            if rank == 0:
                try:  # whatever happens here, rank 0 must reach the collective below (the others wait in it)
                    with torch.cuda.stream(stream):
                        csr = gg.rmat_csr(scale, args.edge_factor, device=dev)
                        stream.synchronize()
                        c1 = ess.Context(local_rank, stream=stream)
                        g1 = ess.Graph(csr)
                        for s, full in zip(timed[:4], fulls):
                            d1, _ = ess.bfs(c1, g1, s, lb="merge_path", direction="optimized")
                            equal = equal and bool(torch.equal(d1, full))
                        del g1, csr, d1
                except Exception as e:
                    equal, failure = False, repr(e)[:300]
            del fulls
            torch.cuda.empty_cache()
            r["equal_single_gpu_bfs"] = bool(all_sum(0 if equal else 1) == 0)
            r["single_gpu_sources_compared"] = len(timed[:4])
            if failure:
                r["single_gpu_check_error"] = failure
        if not args.no_e2e and check_single:
            csr = runner.csr
            h_off, h_col = csr.offsets.cpu().pin_memory(), csr.indices.cpu().pin_memory()
            h_depth = torch.empty(runner.per, dtype=torch.int32).pin_memory()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dist.barrier()
            torch.cuda.synchronize()
            with torch.cuda.stream(stream):
                f0.record(stream)
                for s in timed:
                    csr.offsets.copy_(h_off, non_blocking=True)
                    csr.indices.copy_(h_col, non_blocking=True)
                    runner.bfs(s)
                    runner._fetch_depth()
                    h_depth.copy_(runner.depth_local, non_blocking=True)
                f1.record(stream)
            torch.cuda.synchronize()
            ems = all_max(f0.elapsed_time(f1))
            r["e2e"] = {"value": edges / (ems * 1e-3) / 1e9, "unit": "GTEPS",
                        "h2d_bytes_per_step": int(h_off.numel() * h_off.element_size() + h_col.numel() * 4) * world,
                        "d2h_bytes_per_step": int(runner.n_global * 4), "ms_per_step": ems / steps,
                        "what": "per step and rank: this rank's CSR partition H2D from pinned memory, the partitioned "
                                "BFS, the owned depth slice D2H (bytes summed over ranks); the partition's hint arrays "
                                "are built once (amortised over the steps)"}
        if sssp_steps:
            sv, st, se = 0, 0.0, 0
            runs = []
            with torch.cuda.stream(stream):
                runner.sssp(timed[0])  # warm
                for s in timed[:sssp_steps]:
                    info = runner.sssp(s)
                    n_r, m_r = runner.reached_work_sssp()
                    full = runner.gather_dist()
                    sv += sssp_certificate(runner.csr.offsets, runner.csr.indices, runner.csr.values, full, s,
                                           runner.row_begin)
                    del full
                    t = all_max(info["enact_ms"])
                    st += t
                    se += m_r
                    runs.append({"source": s, "enact_ms": t, "rounds": info["iterations"], "gteps": m_r / t / 1e6,
                                 "exchange": info["exchange"]})
            r["sssp"] = {"runs": runs, "gteps": se / st / 1e6 if st else None,
                         "certificate_violations": all_sum(sv)}
        runner.close()
        del runner
        torch.cuda.empty_cache()
        return r

    main = measure(args.scale, K, W, sssp_steps=2, check_single=True, dump_dir=args.dump_outputs)
    parity_ok = main["certificate_violations"] == 0 and main.get("equal_single_gpu_bfs", True) \
        and main.get("sssp", {}).get("certificate_violations", 0) == 0
    out = {
        "metric": "BFS GTEPS", "value": main["gteps"], "unit": "GTEPS", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": main["ms"] / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "int32", "data": "synthetic",
        "config": workload_config(args.scale, args.edge_factor, main["n"], main["m"], K),
        "implementation": {"advance": "merge_path/optimized", "edge_t_bits": main["offset_bits"],
                           "parallelism": f"1d-vertex-partition x{world}", "exchange_kind": main["exchange_kind"],
                           "levels": main["levels"], "pull_levels": main["pull_levels"]},
        "gpu_launches": main["launches"], "clocks": main["clocks"],
        "parity": {"certificate_violations": main["certificate_violations"], "sources_certified": K,
                   "equal_single_gpu_bfs": main.get("equal_single_gpu_bfs"),
                   "single_gpu_sources_compared": main.get("single_gpu_sources_compared"),
                   "what": "distributed BFS certificate of every timed source (each rank checks its rows against the "
                           "all-gathered depth array) + depths equal to single-GPU ess_bfs on rank 0"},
        "roofline": {"bound": "hbm", "kernel": "partitioned level kernels", "achieved": None, "peak": peak_gbs,
                     "unit": "GB/s", "frac": None, "traffic": None, "peak_source": peak_src,
                     "nvlink_bytes_received_per_rank_per_bfs": main["nvlink_bytes"],
                     "nvlink_time_floor_ms": main["nvlink_bytes"] / 770e9 * 1e3,
                     "nvlink_frac_of_770_gbs": (main["nvlink_bytes"] / 770e9 * 1e3) / (main["ms"] / K),
                     "note": "the single-GPU line carries the kernel roofline; the partitioned step is bound by the "
                             "per-level exchange latency, not by NVLink or HBM bandwidth"},
        "sssp": main.get("sssp"),
    }
    if "e2e" in main:
        out["e2e"] = main["e2e"]
    # ---- secondary workloads: weak scaling (2^24 * 16 generated edges per GPU) and BASELINE config 5 ---------
    if not args.no_extras:
        sec = out.setdefault("other_configs", {})
        if rank == 0:  # not the contract line (that is the single stdout line below): a record of the headline in case a
            # secondary configuration takes the job down
            print("[bench] headline before secondary configs: %.1f GTEPS, %.4f ms/step, parity_ok=%s"
                  % (out["value"], out["ms_per_step"], parity_ok), file=sys.stderr, flush=True)
        try:
            weak_scale = 24 + max(world.bit_length() - 1, 0)
            # the skip decisions must be the same on every rank (measure() is collective): agree on the elapsed time
            if weak_scale != args.scale and all_max(time.time() - T0) < args.extras_budget_s:
                w = measure(weak_scale, min(K, 8), min(W, 3))
                sec["weak_scaling"] = {k: w[k] for k in ("scale", "n", "m", "gteps", "ms", "steps",
                                                         "certificate_violations", "nvlink_bytes")}
                sec["weak_scaling"]["ms_per_step"] = w["ms"] / max(w["steps"], 1)
                parity_ok = parity_ok and w["certificate_violations"] == 0
            if world == 8 and args.scale != 28 and all_max(time.time() - T0) < args.extras_budget_s:
                c5 = measure(28, min(K, 6), 2, sssp_steps=2)
                sec["config5_scale28"] = {k: c5.get(k) for k in ("scale", "n", "m", "gteps", "ms", "steps", "sssp",
                                                                 "certificate_violations", "nvlink_bytes")}
                sec["config5_scale28"]["ms_per_step"] = c5["ms"] / max(c5["steps"], 1)
                parity_ok = parity_ok and c5["certificate_violations"] == 0 \
                    and c5.get("sssp", {}).get("certificate_violations", 0) == 0
        except Exception as e:
            sec["error"] = repr(e)[:300]
    out["parity_ok"] = bool(parity_ok)
    if rank == 0:
        print(json.dumps(out), flush=True)
    return 0 if parity_ok else 3


def main():
    args = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.scale <= 0:
        args.scale = (24 + max(world.bit_length() - 1, 0)) if args.weak else NORTH_STAR_SCALE
    args.scaling = "weak" if args.weak else "strong"
    if args.impl == "reference":
        run_reference(args, rank, world)
        return 0
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        import datetime
        # a rank that dies must not leave the others in a collective for NCCL's default 10 minutes
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank),
                                timeout=datetime.timedelta(seconds=240))
        try:
            return run_distributed(args, rank, world, local_rank)
        finally:
            dist.destroy_process_group()
    return run_single(args, rank, local_rank)


if __name__ == "__main__":
    sys.exit(main())
