"""Latency regime (BASELINE config 5) A/B on ONE GPU holding one shard: the threshold bootstrap
(--bootstrap 1: group-max sample + one filtered slab) against the geometric slab schedule (0), both
replayed from a CUDA graph.  One JSON line per case."""
import argparse, json, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "czech-contriever_b200")]
import torch
from b2ip import Engine

ap = argparse.ArgumentParser()
ap.add_argument("--n-corpus", type=int, default=2_625_000)
ap.add_argument("--d", type=int, default=768)
ap.add_argument("--batches", default="1,64")
ap.add_argument("--k", type=int, default=10)
ap.add_argument("--iters", type=int, default=300)
ap.add_argument("--bootstrap", default="1,0,1,0")
a = ap.parse_args()
dev = torch.device("cuda", 0)

e = Engine(a.d, 0)
e.reserve(a.n_corpus)
CH = 1 << 18
for c0 in range(0, a.n_corpus, CH):
    g = torch.Generator(device=dev).manual_seed(1234 * 1000003 + c0 // CH)
    x = torch.randn((min(CH, a.n_corpus - c0), a.d), generator=g, device=dev)
    x /= x.norm(dim=1, keepdim=True)
    e.add(x)
e.use_torch_stream()
g = torch.Generator(device=dev).manual_seed(4321)
qall = torch.randn((64, a.d), generator=g, device=dev)
qall /= qall.norm(dim=1, keepdim=True)
floor_ms = a.n_corpus * a.d * 2 / 6551e9 * 1e3
ref = {}
for boot in [int(b) for b in a.bootstrap.split(",")]:
    e.set_option("bootstrap", boot)
    for nq in [int(v) for v in a.batches.split(",")]:
        q = qall[:nq].contiguous()
        for _ in range(20):
            D, I = e.search(q, a.k)
        torch.cuda.synchronize()
        dev_ms = 0.0
        t0 = time.perf_counter()
        for _ in range(a.iters):
            D, I = e.search(q, a.k)
            dev_ms += e.stats()["total_ms"]
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3 / a.iters
        st = e.stats()
        e.set_option("graph_timing", 1)
        for _ in range(3):
            e.search(q, a.k)
        sk = e.stats()
        e.set_option("graph_timing", 0)
        same = None
        cand = st["candidates"] / nq
        if nq in ref:
            same = bool(torch.equal(ref[nq][1], I) and torch.equal(ref[nq][0], D))
        else:
            ref[nq] = (D.clone(), I.clone())
        print(json.dumps({"bootstrap": boot, "cand_per_q": round(cand, 1), "rescored_per_q": round(st["rescored"] / nq, 1), "n": a.n_corpus, "nq": nq, "k": a.k, "ms_per_batch": round(wall, 4),
                          "dev_ms": round(dev_ms / a.iters, 4), "floor_ms_16bit": round(floor_ms, 4),
                          "frac_of_floor": round(floor_ms / wall, 4), "graph_mode": st["graph_mode"],
                          "launches": st["total_launches"], "coarse_launches": st["coarse_launches"], "slabs": st["slabs"],
                          "coarse_ms": round(sk["coarse_ms"], 4), "refresh_ms": round(sk["refresh_ms"], 4),
                          "finalize_ms": round(sk["finalize_ms"], 4), "fallback": st["fallback_queries"],
                          "same_as_first": same}), flush=True)
