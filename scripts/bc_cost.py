"""What betweenness centrality costs per source next to the BFS it starts from, one GPU.

Workloads: symmetric Kronecker graphs (edge factor 16, bench.py's generator) at scale-24 and scale-26, `--sources`
pick_sources sources each. Both calls are warmed up, then every round times ess.bc(sources=[s]) and ess.bfs(s,
merge_path, optimized) with CUDA events on the context's stream, in an order that flips every round. Every timed bc
is checked on the device by certificate(). Reported per workload: ms per source of each call, the BFS share of bc, the
edges the two gathers walked per second, and the byte floor of those gathers: two passes over the column indices,
at least 8 · m bytes per source, over the HBM bandwidth of the data sheet (7.7 TB/s). Prints one JSON line with the
card's name and power limit; exits 1 on any failed certificate:

  python scripts/bc_cost.py --out profiles/r03c_bc_cost.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INT_MAX = 2**31 - 1
HBM_BYTES_PER_S = 7.7e12


def certificate(bc, depth, source, degree):
    """Device check of a single-source bc (scale 1) against that source's BFS depths, in torch:
    rel_err       |Σ bc (float64) - Σ_{t reached, t != s} (depth[t] - 1)| / that sum: every interior vertex of every
                  shortest path is counted once, so the dependencies add up to the hops minus one of each target;
    negative      entries below 0;
    leaf_nonzero  non-zero entries at vertices with at most one distinct neighbour other than themselves (`degree`
                  must count exactly those), which lie inside no shortest path."""
    import torch
    n = depth.numel()
    bc = bc[:n]
    reached = depth != INT_MAX
    reached[source] = False
    want = float((depth[reached].double() - 1.0).sum().item())
    got = float(bc.double().sum().item())
    return {"rel_err": abs(got - want) / max(want, 1.0), "negative": int((bc < 0).sum().item()),
            "leaf_nonzero": int(((degree <= 1) & (bc != 0)).sum().item()), "dependency_sum": want}


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return torch.cuda.get_device_name(), q.stdout.strip() or "unknown"


def measure(ess, torch, stream, name, csr, sources, rounds):
    with torch.cuda.stream(stream):
        ctx = ess.Context(0, stream=stream)
        g = ess.Graph(csr)
        out = torch.empty(csr.n, dtype=torch.float32, device="cuda")
        depth = torch.empty(csr.n, dtype=torch.int32, device="cuda")
        degree = csr.degrees()  # rmat_csr graphs are simple: the degree counts distinct neighbours
        ess.bc(ctx, g, [sources[0]], out=out)  # warm
        ess.bfs(ctx, g, sources[0], lb="merge_path", direction="optimized", out=depth)  # warm
    stream.synchronize()
    run = {"bc": lambda s: ess.bc(ctx, g, [s], out=out),
           "bfs": lambda s: ess.bfs(ctx, g, s, lb="merge_path", direction="optimized", out=depth)}
    ms = {k: 0.0 for k in run}
    edges, levels, failed, worst = 0, 0, 0, 0.0
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
                if k == "bc":
                    edges += info["edges_gathered"]
                    levels = max(levels, info["levels"])
            with torch.cuda.stream(stream):  # both buffers now hold source s
                c = certificate(out, depth, s, degree)
            stream.synchronize()
            worst = max(worst, c["rel_err"])
            failed += int(c["rel_err"] > 1e-6 or c["negative"] or c["leaf_nonzero"])
    calls = rounds * len(sources)
    per = {k: ms[k] / calls for k in ms}
    gathered = edges / calls
    g.close()
    ctx.close()
    return {"workload": name, "n": csr.n, "m": csr.m, "sources": len(sources), "rounds": rounds,
            "ms_bc_per_source": round(per["bc"], 4), "ms_bfs_per_source": round(per["bfs"], 4),
            "bfs_pct_of_bc": round(100.0 * per["bfs"] / per["bc"], 2), "levels_max": levels,
            "edges_gathered_per_source": int(gathered),
            "gathered_edges_per_s_1e9": round(gathered / (per["bc"] * 1e-3) / 1e9, 2),
            "index_bytes_floor_per_source": 8 * csr.m,
            "floor_ms_at_7p7TBps": round(8 * csr.m / HBM_BYTES_PER_S * 1e3, 4),
            "certificate_max_rel_err": worst, "failed_certificates": failed}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", help="also write the JSON line to this file")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--sources", type=int, default=8)
    ap.add_argument("--scales", default="24,26")
    args = ap.parse_args()
    import torch
    sys.path.insert(0, ROOT)
    import essentials_b200 as ess
    from essentials_b200 import graphgen as gg
    assert torch.cuda.is_available(), "bc_cost.py measures on a GPU"
    stream = torch.cuda.Stream()
    name, power = card()
    res = []
    for scale in (int(x) for x in args.scales.split(",")):
        with torch.cuda.stream(stream):  # built on the stream the measurement runs on, so nothing races the build
            kron = gg.rmat_csr(scale, 16, device="cuda")
        stream.synchronize()  # pick_sources reads the degrees on the default stream
        res.append(measure(ess, torch, stream, f"kron scale-{scale} ef-16 symmetric", kron,
                           gg.pick_sources(kron, args.sources), args.rounds))
        del kron
        torch.cuda.empty_cache()
    line = json.dumps({"metric": "BC cost per source", "device": name, "power_limit": power, "results": res})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    sys.exit(0 if all(r["failed_certificates"] == 0 for r in res) else 1)


if __name__ == "__main__":
    main()
