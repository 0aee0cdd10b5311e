"""Range search next to k-NN search on the same corpus and queries.

Builds a seeded, device-resident, L2-normalised fp32 corpus (a 2.6M-row shard, and with --full the
21M-row corpus when the GPU has the memory), takes 1,000 seeded queries, sets the radius to the median
of the queries' 100th scores (so a query gets about 100 rows), and alternates `search(k=100)` and
`range_search(radius)`.  Prints one JSON line per corpus: ms per call (median over --iters), the
coarse and finalize / drain kernel times, candidates and rescored rows per query, and the GPU's name
and power limit read in the same run.

    python tools/range_bench.py [--full] [--iters 7] [--out OUT_DIR/range_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "czech-contriever_b200"))


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


def run(n, d, nq, k, iters):
    import numpy as np
    import torch
    e = corpus(n, d, seed=1234)
    g = torch.Generator(device="cuda").manual_seed(4321)
    q = torch.randn((nq, d), generator=g, device="cuda")
    q /= q.norm(dim=1, keepdim=True)
    D, _ = e.search(q, k)
    radius = float(np.float32(D[:, -1].median().item()))
    e.range_search(q, radius)                  # warm-up of both shapes
    rec = {"knn": [], "range": []}
    for _ in range(iters):
        ms, _ = timed(lambda: e.search(q, k))
        rec["knn"].append((ms, e.stats()))
        ms, ans = timed(lambda: e.range_search(q, radius))
        rec["range"].append((ms, e.stats()))
    lims = ans[0].cpu().numpy()

    def summary(rows):
        i = int(np.argsort([r[0] for r in rows])[len(rows) // 2])
        ms, st = rows[i]
        return {"ms_per_call": round(ms, 3), "total_ms": round(st["total_ms"], 3),
                "coarse_ms": round(st["coarse_ms"], 3), "finalize_ms": round(st["finalize_ms"], 3),
                "refresh_ms": round(st["refresh_ms"], 3), "slabs": st["slabs"],
                "candidates_per_query": round(st["candidates"] / nq, 1),
                "rescored_per_query": round(st["rescored"] / nq, 1),
                "fallback_queries": st["fallback_queries"], "bound_violations": st["bound_violations"]}

    out = {"rows": n, "d": d, "nq": nq, "k": k, "radius": radius,
           "mean_results_per_query": round(float(lims[-1]) / nq, 1),
           "min_results": int(np.diff(lims).min()), "max_results": int(np.diff(lims).max()),
           "knn": summary(rec["knn"]), "range": summary(rec["range"])}
    e.close()
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--full", action="store_true", help="also the 21M-row corpus (needs ~100 GB free)")
    ap.add_argument("--iters", type=int, default=7)
    ap.add_argument("--nq", type=int, default=1000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("range_bench: no CUDA device (this measures the B200 engine; there is no CPU path)")
    name, power = gpu_info()
    sizes = [2_600_000]
    if a.full:
        free, _ = torch.cuda.mem_get_info(0)
        if free > 21_000_000 * 768 * 6 * 1.1:      # fp32 master rows + 16-bit shadow
            sizes.append(21_000_000)
    lines = []
    for n in sizes:
        res = run(n, 768, a.nq, 100, a.iters)
        res.update({"gpu": name, "power_limit": power})
        lines.append(json.dumps(res))
        print(lines[-1], flush=True)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
