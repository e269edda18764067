"""What the BFS tree costs: ess.bfs against ess.bfs_tree on the same sources, one GPU.

Workloads: the headline graph (Kronecker scale-26, edge factor 16, merge_path, direction-optimised) and Kronecker
scale-24 with merge_path forward (push only). Per workload, 16 pick_sources sources; both entry points are warmed up
on two other sources, then each source runs ess.bfs and ess.bfs_tree back to back (the order flips every round), 3
rounds, each call timed with CUDA events on the context's stream (problem reset + enact, as bench.py times a step).
Every tree is checked on the device by tree_violations() and every depth array must equal ess.bfs's bit for bit.
Prints one JSON line with the card's name and power limit:

  python scripts/bfs_tree_cost.py --out profiles/r03a_bfs_tree_cost.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INT32_MAX = 2**31 - 1


def tree_violations(offsets, indices, source, depth, pred, chunk=1 << 26):
    """Device check of a BFS tree against its depth array; every count is 0 for a valid tree.
    source:    pred[source] != source
    unreached: vertices where (pred == -1) differs from (depth == INT32_MAX)
    range:     other reached vertices whose parent is outside [0, n)
    depth:     ... whose parent's depth is not depth - 1
    edge:      ... whose parent u has no edge u -> v in the CSR (one pass over the edges, `chunk` at a time)."""
    import torch
    n, m = offsets.numel() - 1, indices.numel()
    out = {"source": int(pred[source].item() != source)}
    unreached = depth == INT32_MAX
    out["unreached"] = int(((pred == -1) != unreached).sum().item())
    rest = ~unreached
    rest[source] = False
    v = rest.nonzero().squeeze(1)
    u = pred[v].long()
    ok = (u >= 0) & (u < n)
    out["range"] = int((~ok).sum().item())
    v, u = v[ok], u[ok]
    out["depth"] = int((depth[u] != depth[v] - 1).sum().item())
    # an edge r -> c of the CSR proves the parent of c when pred[c] == r
    hit = torch.zeros(n, dtype=torch.bool, device=depth.device)
    off = offsets.long()
    for e0 in range(0, m, chunk):
        e1 = min(m, e0 + chunk)
        rows = torch.searchsorted(off, torch.arange(e0, e1, device=depth.device), right=True) - 1
        cols = indices[e0:e1].long()
        hit[cols[pred[cols].long() == rows]] = True
    out["edge"] = int((~hit[v]).sum().item())
    return out


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return torch.cuda.get_device_name(), q.stdout.strip() or "unknown"


def measure(ess, gg, torch, stream, name, scale, lb, direction, rounds, count):
    with torch.cuda.stream(stream):
        csr = gg.rmat_csr(scale, 16, device="cuda")
        ctx = ess.Context(0, stream=stream)
        g = ess.Graph(csr)
        depth = torch.empty(csr.n, dtype=torch.int32, device="cuda")
        tdepth = torch.empty_like(depth)
        pred = torch.empty_like(depth)
    stream.synchronize()
    srcs = gg.pick_sources(csr, count + 2)
    warm, timed = srcs[:2], srcs[2:]
    deg = csr.degrees().long()
    run = {"bfs": lambda s: ess.bfs(ctx, g, s, lb=lb, direction=direction, out=depth),
           "bfs_tree": lambda s: ess.bfs_tree(ctx, g, s, lb=lb, direction=direction, out=tdepth, pred_out=pred)}
    with torch.cuda.stream(stream):
        for s in warm:
            for f in run.values():
                f(s)
    stream.synchronize()
    ms = {k: 0.0 for k in run}
    edges, bad, mismatched, violations = 0, 0, 0, {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(rounds):
        order = list(run) if r % 2 == 0 else list(run)[::-1]
        for s in timed:
            for k in order:
                with torch.cuda.stream(stream):
                    e0.record(stream)
                    run[k](s)
                    e1.record(stream)
                stream.synchronize()
                ms[k] += e0.elapsed_time(e1)
            with torch.cuda.stream(stream):
                v = tree_violations(csr.offsets, csr.indices, s, tdepth, pred)
                mismatched += int(not torch.equal(depth, tdepth))
                if r == 0:
                    edges += int(deg[depth != INT32_MAX].sum().item())
            stream.synchronize()
            bad += int(any(v.values()))
            for key, c in v.items():
                violations[key] = violations.get(key, 0) + c
    calls = rounds * len(timed)
    per = {k: ms[k] / calls for k in ms}
    g.close()
    ctx.close()
    return {"workload": name, "n": csr.n, "m": csr.m, "lb": lb, "direction": direction, "sources": len(timed),
            "rounds": rounds, "ms_bfs": round(per["bfs"], 4), "ms_bfs_tree": round(per["bfs_tree"], 4),
            "diff_ms": round(per["bfs_tree"] - per["bfs"], 4),
            "diff_pct": round(100.0 * (per["bfs_tree"] - per["bfs"]) / per["bfs"], 2),
            "gteps_bfs": round(edges / len(timed) / (per["bfs"] * 1e-3) / 1e9, 1),
            "gteps_bfs_tree": round(edges / len(timed) / (per["bfs_tree"] * 1e-3) / 1e9, 1),
            "invalid_trees": bad, "violations": violations, "depth_mismatches": mismatched}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", help="also write the JSON line to this file")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--sources", type=int, default=16)
    ap.add_argument("--scales", default="26,24", help="headline scale, push-only scale")
    args = ap.parse_args()
    import torch
    sys.path.insert(0, ROOT)
    import essentials_b200 as ess
    from essentials_b200 import graphgen as gg
    assert torch.cuda.is_available(), "bfs_tree_cost.py measures on a GPU"
    big, push = (int(x) for x in args.scales.split(","))
    stream = torch.cuda.Stream()
    name, power = card()
    res = [measure(ess, gg, torch, stream, f"kron scale-{big} ef-16", big, "merge_path", "optimized", args.rounds,
                   args.sources),
           measure(ess, gg, torch, stream, f"kron scale-{push} ef-16", push, "merge_path", "forward", args.rounds,
                   args.sources)]
    line = json.dumps({"metric": "BFS tree cost", "device": name, "power_limit": power, "results": res})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    ok = all(r["invalid_trees"] == 0 and r["depth_mismatches"] == 0 for r in res)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
