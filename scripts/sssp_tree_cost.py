"""What the SSSP tree costs next to the SSSP run it follows, one GPU.

Workloads: bench.py's two SSSP lines. Weighted Kronecker scale-24 (edge factor 16, symmetric pair-hash weights in
[1, 64)) with ess.sssp_delta from `--sources` pick_sources sources, and the 4900 x 4900 grid (pair-hash weights) with
ess.sssp_near_far from vertex 0. Each source's distances are computed once and kept; both calls are warmed up, then
every round times ess.sssp (into a second buffer) and ess.sssp_tree (on the kept distances) with CUDA events on the
context's stream, in an order that flips every round. Every tree is checked on the device by sssp_tree_violations(),
and every timed SSSP result must equal the kept distances bit for bit. Prints one JSON line with the card's name and
power limit; exits 1 on any invalid tree or distance mismatch:

  python scripts/sssp_tree_cost.py --out profiles/r03b_sssp_tree_cost.json
"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLT_MAX = 3.4028234663852886e38


def sssp_tree_violations(offsets, indices, values, source, dist, pred, chunk=1 << 26):
    """Check of an SSSP tree against its distance array, in torch (device or host tensors); every count is 0 for a
    valid tree.
    source:    pred[source] != source
    unreached: vertices where (pred == -1) differs from (dist == FLT_MAX)
    range:     other reached vertices whose parent is outside [0, n)
    edge:      ... whose parent u has no tight edge u -> v in the CSR (dist[u] + w == dist[v] in float32, w = 1 without
               values; one pass over the edges, `chunk` at a time)
    cycle:     reached vertices that ceil(log2 n) + 1 pointer-jumping steps over pred do not take to the source."""
    import torch
    n, m = offsets.numel() - 1, indices.numel()
    dev = dist.device
    pred = pred[:n].long()
    dist = dist[:n]
    out = {"source": int(pred[source].item() != source)}
    reached = dist != FLT_MAX
    out["unreached"] = int(((pred == -1) != ~reached).sum().item())
    rest = reached.clone()
    rest[source] = False
    in_range = (pred >= 0) & (pred < n)
    out["range"] = int((rest & ~in_range).sum().item())
    # an edge r -> c of the CSR proves the parent of c when pred[c] == r and the edge is tight
    hit = torch.zeros(n, dtype=torch.bool, device=dev)
    off = offsets.long()
    for e0 in range(0, m, chunk):
        e1 = min(m, e0 + chunk)
        rows = torch.searchsorted(off, torch.arange(e0, e1, device=dev), right=True) - 1
        cols = indices[e0:e1].long()
        w = values[e0:e1] if values is not None else torch.ones(e1 - e0, dtype=torch.float32, device=dev)
        tight = (dist[rows] != FLT_MAX) & ((dist[rows] + w) == dist[cols])
        ok = tight & (pred[cols] == rows)
        hit[cols[ok]] = True
    out["edge"] = int((rest & in_range & ~hit).sum().item())
    # pointer jumping: out-of-range parents and unreached vertices point at themselves
    anc = torch.where(rest & in_range, pred, torch.arange(n, device=dev))
    anc[source] = source
    for _ in range(math.ceil(math.log2(max(n, 2))) + 1):
        anc = anc[anc]
    out["cycle"] = int((reached & (anc != source)).sum().item())
    return out


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return torch.cuda.get_device_name(), q.stdout.strip() or "unknown"


def measure(ess, torch, stream, name, csr, engine, sources, rounds):
    with torch.cuda.stream(stream):
        ctx = ess.Context(0, stream=stream)
        g = ess.Graph(csr)
        scratch = torch.empty(csr.n, dtype=torch.float32, device="cuda")
        pred = torch.empty(csr.n, dtype=torch.int32, device="cuda")
    sssp = getattr(ess, engine)
    kept = {}
    with torch.cuda.stream(stream):
        for s in sources:
            kept[s], _ = sssp(ctx, g, s)
            sssp(ctx, g, s, out=scratch)  # warm
            ess.sssp_tree(ctx, g, s, kept[s], pred_out=pred)  # warm
    stream.synchronize()
    run = {"sssp": lambda s: sssp(ctx, g, s, out=scratch),
           "tree": lambda s: ess.sssp_tree(ctx, g, s, kept[s], pred_out=pred)}
    ms = {k: 0.0 for k in run}
    bad, mismatched, violations, flat_rounds, flat_vertices = 0, 0, {}, 0, 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(rounds):
        order = list(run) if r % 2 == 0 else list(run)[::-1]
        for s in sources:
            for k in order:
                with torch.cuda.stream(stream):
                    e0.record(stream)
                    _, info = run[k](s)
                    e1.record(stream)
                stream.synchronize()
                ms[k] += e0.elapsed_time(e1)
                if k == "tree":
                    flat_rounds = max(flat_rounds, info["flat_rounds"])
                    flat_vertices = max(flat_vertices, info["flat_vertices"])
            with torch.cuda.stream(stream):
                v = sssp_tree_violations(csr.offsets, csr.indices, csr.values, s, kept[s], pred)
                mismatched += int(not torch.equal(scratch, kept[s]))
            stream.synchronize()
            bad += int(any(v.values()))
            for key, c in v.items():
                violations[key] = violations.get(key, 0) + c
    calls = rounds * len(sources)
    per = {k: ms[k] / calls for k in ms}
    g.close()
    ctx.close()
    return {"workload": name, "n": csr.n, "m": csr.m, "engine": engine, "sources": len(sources), "rounds": rounds,
            "ms_sssp": round(per["sssp"], 4), "ms_tree": round(per["tree"], 4),
            "tree_pct_of_sssp": round(100.0 * per["tree"] / per["sssp"], 2),
            "tree_edges_per_s": round(csr.m / (per["tree"] * 1e-3) / 1e9, 2),
            "flat_rounds_max": flat_rounds, "flat_vertices_max": flat_vertices,
            "invalid_trees": bad, "violations": violations, "dist_mismatches": mismatched}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", help="also write the JSON line to this file")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--sources", type=int, default=8, help="Kronecker sources")
    ap.add_argument("--scale", type=int, default=24)
    ap.add_argument("--grid", type=int, default=4900)
    args = ap.parse_args()
    import torch
    sys.path.insert(0, ROOT)
    import essentials_b200 as ess
    from essentials_b200 import graphgen as gg
    assert torch.cuda.is_available(), "sssp_tree_cost.py measures on a GPU"
    stream = torch.cuda.Stream()
    name, power = card()
    with torch.cuda.stream(stream):  # built on the stream the measurement runs on, so nothing races the build
        kron = gg.rmat_csr(args.scale, 16, weights="hash", device="cuda")
    stream.synchronize()  # pick_sources reads the degrees on the default stream
    res = [measure(ess, torch, stream, f"kron scale-{args.scale} ef-16 hash weights", kron, "sssp_delta",
                   gg.pick_sources(kron, args.sources), args.rounds)]
    del kron
    torch.cuda.empty_cache()
    with torch.cuda.stream(stream):
        grid = gg.grid_csr(args.grid, args.grid, device="cuda")
    stream.synchronize()
    res.append(measure(ess, torch, stream, f"grid {args.grid}x{args.grid} hash weights", grid, "sssp_near_far", [0],
                       args.rounds))
    line = json.dumps({"metric": "SSSP tree cost", "device": name, "power_limit": power, "results": res})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    ok = all(r["invalid_trees"] == 0 and r["dist_mismatches"] == 0 for r in res)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
