"""Filtered k-NN search next to the unfiltered search on the same corpus and queries.

Builds a seeded, device-resident, L2-normalised fp32 corpus (a 2.6M-row shard, and with --full the
21M-row corpus when the GPU has the memory) and runs two query shapes, nq = 1000 / k = 100 and
nq = 64 / k = 10, at allowed fractions 1 (the unfiltered call), 1 (an all-ones mask), 0.5, 0.1, 0.01
and 0.001.  The masks are seeded random device tensors; the calls of one shape alternate over the
fractions, --iters rounds.  Prints one JSON line per (corpus, shape): per fraction the median ms
per call, the coarse, refresh and finalize kernel times, candidates and fallbacks per query, and
the GPU's name and power limit read in the same run.

    python tools/filter_bench.py [--full] [--iters 9] [--out OUT_DIR/filter_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "czech-contriever_b200"))

FRACTIONS = ["none", 1.0, 0.5, 0.1, 0.01, 0.001]     # "none" = the unfiltered call
SHAPES = [(1000, 100), (64, 10)]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception as exc:                   # (the numbers below still carry torch's device name)
        import torch
        return torch.cuda.get_device_name(0), f"unknown ({exc})"


def corpus(n, d, seed):
    import torch
    import b2ip
    e = b2ip.Engine(d, 0)
    e.reserve(n)
    g = torch.Generator(device="cuda").manual_seed(seed)
    for c0 in range(0, n, 1 << 20):
        x = torch.randn((min(1 << 20, n - c0), d), generator=g, device="cuda")
        x /= x.norm(dim=1, keepdim=True)
        e.add(x)
        del x
    return e


def timed(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def run(e, n, d, nq, k, iters):
    import numpy as np
    import torch
    g = torch.Generator(device="cuda").manual_seed(4321 + nq)
    q = torch.randn((nq, d), generator=g, device="cuda")
    q /= q.norm(dim=1, keepdim=True)
    masks = {f: (None if f == "none" else torch.rand(n, generator=g, device="cuda") < f) for f in FRACTIONS}
    for f in FRACTIONS:                        # warm-up (and graph capture) of every call
        e.search(q, k, allowed=masks[f])
    rec = {f: [] for f in FRACTIONS}
    for _ in range(iters):
        for f in FRACTIONS:
            ms, _ = timed(lambda: e.search(q, k, allowed=masks[f]))
            rec[f].append((ms, e.stats()))

    def summary(rows):
        i = int(np.argsort([r[0] for r in rows])[len(rows) // 2])
        ms, st = rows[i]
        return {"ms_per_call": round(ms, 3), "total_ms": round(st["total_ms"], 3),
                "coarse_ms": round(st["coarse_ms"], 3), "refresh_ms": round(st["refresh_ms"], 3),
                "finalize_ms": round(st["finalize_ms"], 3), "slabs": st["slabs"],
                "candidates_per_query": round(st["candidates"] / nq, 1),
                "fallbacks_per_query": round(st["fallback_queries"] / nq, 4),
                "graph_mode": st["graph_mode"], "bound_violations": st["bound_violations"]}

    return {"rows": n, "d": d, "nq": nq, "k": k,
            "by_fraction": {("unfiltered" if f == "none" else f"mask_{f}"): summary(rec[f]) for f in FRACTIONS}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--full", action="store_true", help="also the 21M-row corpus (needs ~100 GB free)")
    ap.add_argument("--iters", type=int, default=9)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("filter_bench: no CUDA device (this measures the B200 engine; there is no CPU path)")
    name, power = gpu_info()
    sizes = [2_600_000]
    if a.full:
        free, _ = torch.cuda.mem_get_info(0)
        if free > 21_000_000 * 768 * 6 * 1.1:      # fp32 master rows + 16-bit shadow
            sizes.append(21_000_000)
    lines = []
    for n in sizes:
        e = corpus(n, 768, seed=1234)
        # per-kernel times of the small batch come from event records inside its CUDA graph
        e.set_option("graph_timing", 1)
        for nq, k in SHAPES:
            res = run(e, n, 768, nq, k, a.iters)
            res.update({"gpu": name, "power_limit": power})
            lines.append(json.dumps(res))
            print(lines[-1], flush=True)
        e.close()
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
