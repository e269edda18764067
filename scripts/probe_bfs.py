"""Quick perf probe (development aid): BFS variants on a Kronecker graph, enact() ms and GTEPS."""
import argparse
import time

import numpy as np
import torch

import essentials_b200 as ess
from essentials_b200 import graphgen as gg

ap = argparse.ArgumentParser()
ap.add_argument("--scale", type=int, default=24)
ap.add_argument("--sources", type=int, default=4)
ap.add_argument("--variants", default="block_mapped:forward,merge_path:forward,bucketing:forward,"
                                      "block_mapped:optimized,merge_path:optimized,bucketing:optimized")
ap.add_argument("--sssp", action="store_true")
ap.add_argument("--pull-variants", default="")
ap.add_argument("--hints", default="1")
ap.add_argument("--alphas", default="0")
ap.add_argument("--betas", default="0")
ap.add_argument("--engines", default="1", help="comma list of advance_engine values: 1 quad engine, 0 scalar kernels")
args = ap.parse_args()

t = time.time()
csr = gg.rmat_csr(args.scale, device="cuda", weights="hash" if args.sssp else "none")
torch.cuda.synchronize()
print(f"graph {csr.name}: n={csr.n} m={csr.m} offsets={csr.offsets.dtype} built in {time.time()-t:.1f}s", flush=True)
ctx = ess.Context(0)
g = ess.Graph(csr)
srcs = gg.pick_sources(csr, args.sources)
deg = csr.degrees().long()
base = None
runs = [(v, None) for v in args.variants.split(",")]
if args.pull_variants:
    runs = [(v, int(pv)) for pv in args.pull_variants.split(",") for v in args.variants.split(",")]
runs = [(v, pv, int(h), float(a), float(b), eng) for eng in args.engines.split(",") for (v, pv) in runs
        for h in args.hints.split(",") for a in args.alphas.split(",") for b in args.betas.split(",")]
for variant, pv, hints, alpha, beta, eng in runs:
    lb, direction = variant.split(":")
    ess.tune("pull_hints", hints)
    ess.tune("advance_engine", int(eng))
    variant = f"{variant}/eng{eng}/h{hints}/a{alpha:g}/b{beta:g}"
    for s in srcs:
        ctx.profile(True)
        depth, info = ess.bfs(ctx, g, s, lb=lb, direction=direction, alpha=alpha, beta=beta)
        prof = ctx.profile_read()
        ctx.profile(False)
        reached = depth != 2**31 - 1
        m_r = int(deg[reached].sum())
        if base is None:
            base = {}
        if s in base:
            assert torch.equal(base[s], depth), f"{variant} differs from the first variant at source {s}"
        else:
            base[s] = depth.clone()
        print(f"{variant:40s} src={s:9d} enact={info['enact_ms']:9.3f} ms  levels={info['iterations']:3d} "
              f"pull={info['pull_steps']}  reached={int(reached.sum())}  GTEPS={m_r/info['enact_ms']/1e6:8.2f}  "
              + " ".join(f"{k}={v[0]:.3f}ms/{v[1]}" for k, v in prof.items() if v[1])
              + f" pullV={info['pull_vertices']} pullE={info['pull_edges']} pushV={info['push_vertices']} pushE={info['push_edges']}",
              flush=True)
if args.sssp:
    for lb in ("block_mapped", "merge_path", "bucketing"):
        for s in srcs[:2]:
            dist, info = ess.sssp(ctx, g, s, lb=lb)
            reached = dist < 3e38
            m_r = int(deg[reached].sum())
            print(f"sssp {lb:22s} src={s:9d} enact={info['enact_ms']:9.3f} ms iters={info['iterations']} "
                  f"GTEPS={m_r/info['enact_ms']/1e6:8.2f}", flush=True)
