"""Perf + parity probe for BASELINE configs 3 (SSSP on a 2-D grid) and 4 (PageRank on directed RMAT)."""
import argparse
import time

import numpy as np
import torch

import essentials_b200 as ess
import oracle
from essentials_b200 import graphgen as gg

ap = argparse.ArgumentParser()
ap.add_argument("--grid", type=int, default=4900)
ap.add_argument("--pr-scale", type=int, default=25)
ap.add_argument("--skip-sssp", action="store_true")
ap.add_argument("--skip-pr", action="store_true")
ap.add_argument("--check", action="store_true", help="compare with the CPU oracle (slow at full size)")
ap.add_argument("--lbs", default="thread_mapped,block_mapped,merge_path,bucketing")
args = ap.parse_args()
ctx = ess.Context(0)

if not args.skip_sssp:
    t = time.time()
    csr = gg.grid_csr(args.grid, args.grid, device="cuda")
    g = ess.Graph(csr)
    print(f"grid {args.grid}^2: n={csr.n} m={csr.m} built in {time.time()-t:.1f}s", flush=True)
    want = None
    if args.check:
        off, col, val = csr.host()
        want, cpu_ms = oracle.sssp(off, col, val, 0, return_ms=True)
        print(f"cpu oracle sssp: {cpu_ms/1e3:.2f} s  ({csr.m/cpu_ms/1e6:.4f} GTEPS)", flush=True)
    for lb in args.lbs.split(","):
        ctx.profile(True)
        dist, info = ess.sssp(ctx, g, 0, lb=lb)
        prof = ctx.profile_read()
        ctx.profile(False)
        ok = "" if want is None else f" bit-exact={np.array_equal(dist.cpu().numpy(), want)}"
        print(f"sssp {lb:14s} enact={info['enact_ms']:10.2f} ms iters={info['iterations']} "
              f"GTEPS={csr.m/info['enact_ms']/1e6:.4f}{ok}  "
              + " ".join(f"{k}={v[0]:.1f}ms/{v[1]}" for k, v in prof.items() if v[1]), flush=True)
    for delta in (0.0, 512.0, 2048.0, 8192.0):
        dist, info = ess.sssp_near_far(ctx, g, 0, delta=delta)
        ok = "" if want is None else f" bit-exact={np.array_equal(dist.cpu().numpy(), want)}"
        print(f"sssp near_far delta={delta:6.1f} enact={info['enact_ms']:10.2f} ms levels={info['levels']} "
              f"splits={info['splits']} relaxations={info['relaxations']} ({info['relaxations']/csr.m:.2f} x m) "
              f"GTEPS={csr.m/info['enact_ms']/1e6:.4f}{ok}", flush=True)
    del g, csr

if not args.skip_pr:
    t = time.time()
    csr = gg.rmat_csr(args.pr_scale, symmetric=False, weights="ones", device="cuda")
    csc = ess.transpose(csr)
    g = ess.Graph(csr, csc=csc)
    torch.cuda.synchronize()
    print(f"rmat directed scale-{args.pr_scale}: n={csr.n} m={csr.m} built in {time.time()-t:.1f}s", flush=True)
    runs = [("pull", "block_mapped", True)] + [(lb, lb, False) for lb in args.lbs.split(",")]
    res = {}
    for name, lb, pull in runs:
        p, info = ess.pagerank(ctx, g, lb=lb, pull=pull)
        res[name] = p.clone()
        it = info["iterations"]
        print(f"pr {name:14s} enact={info['enact_ms']:10.2f} ms iters={it} ms/iter={info['enact_ms']/it:.3f} "
              f"GTEPS={csr.m*it/info['enact_ms']/1e6:.2f} sum={float(p.double().sum()):.6f}", flush=True)
    base = res["pull"].double()
    for name, p in res.items():
        rel = ((p.double() - base).abs().sum() / base.sum()).item()
        print(f"  {name}: rel-L1 vs pull {rel:.3e}", flush=True)
    if args.check:
        off, col, val = csr.host()
        p_gpu, info = ess.pagerank(ctx, g, pull=True, max_iterations=5)
        want, _ = oracle.pagerank(off, col, val, force_iters=5)
        got = p_gpu.cpu().numpy().astype(np.float64)
        print("pr pull vs oracle after 5 iterations: max rel err", float(np.max(np.abs(got - want) / want)), flush=True)
