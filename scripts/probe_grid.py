"""Perf probe (development aid): SSSP on the 4900 x 4900 grid through execute_near_far — bucket widths."""
import argparse

import numpy as np
import torch

import essentials_b200 as ess
from essentials_b200 import graphgen as gg

ap = argparse.ArgumentParser()
ap.add_argument("--grid", type=int, default=4900)
ap.add_argument("--deltas", default="0,64,128,256,512,1024")
ap.add_argument("--reps", type=int, default=2)
args = ap.parse_args()
ctx = ess.Context(0)
csr = gg.grid_csr(args.grid, args.grid, device="cuda")
g = ess.Graph(csr)
base = None
for delta in [float(x) for x in args.deltas.split(",")]:
    for rep in range(args.reps):
        dist, info = ess.sssp_near_far(ctx, g, 0, delta=delta)
    if base is None:
        base = dist.clone()
    same = bool(torch.equal(base, dist))
    print(f"delta={delta:7.1f} enact={info['enact_ms']:9.2f} ms levels={info['levels']} "
          f"splits={info['splits']} us/level={1e3*info['enact_ms']/max(info['levels'],1):.2f} "
          f"relax={info['relaxations']/csr.m:.2f}x m GTEPS={csr.m/info['enact_ms']/1e6:.3f} equal={same}", flush=True)
