#!/usr/bin/env python
"""bench.py -- exact top-k inner-product search throughput (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b2ip|reference]

One "step" = one pass of the hot path over one batch of synthetic queries: all `n_queries`
queries against the whole row-sharded corpus (local tcgen05 scoring + fused filter + fp32
rescore per GPU, then the peer-direct exchange + merge when N > 1).  Default workload = BASELINE
config 3: 21M x 768 fp32 L2-normalised synthetic corpus, 100k queries, k = 100 (fits one B200:
64.5 GB fp32 master + 32.3 GB bf16 shadow).  The corpus is fixed as N grows -> "strong".

Prints ONE JSON line on rank 0:
  value            queries/s with the queries resident in HBM (K timed steps, CUDA events, max over ranks)
  e2e              the same through the reference-facing C-ABI call with PAGEABLE host buffers
                   (numpy in / numpy out, H2D and D2H inside the timed region); at N > 1 through
                   `ShardedIndex.search_host` (each rank uploads the queries and downloads its
                   slice of the result into one host array shared by the ranks)
  e2e_search_knn   wall time of the drop-in `Indexer.search_knn` (reference src/index.py:34-46,
                   the region passage_retrieval.py:188-190 times): pageable float16 queries ->
                   list of (list[str], float32 row); at N > 1 from ONE process driving all N GPUs
                   (`Indexer(device="all")`, what an unmodified reference driver uses)
  roofline         the tcgen05 scoring kernel against the measured bf16 peak
  cpu_baseline     the faiss-equivalent CPU oracle on the box's host cores: a query subset
                   against the FULL corpus (BASELINE.md 3), N = 1 only
  parity_probe     fp64 brute force over every rank's shard for 32 of the timed queries,
                   compared tie-aware with the timed result (pass / fail)
  secondary        BASELINE configs C5 (batch 64, k = 10: HBM roofline), C2 and C4, each with
                   its own roofline -- so the driver's records hold them at every N
`--impl reference` times the CPU implementation alone (rank 0 only under torchrun).
`--workload c2|c4|c5` makes another BASELINE config the primary line (for profiles/).
`--dump-outputs DIR` writes the last timed step's answer (see `dump_outputs`) so that two builds
can be compared output for output: the inputs are seeded, identical from run to run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True     # the benchmark writes nothing into the tree it runs from
os.environ.setdefault("OMP_WAIT_POLICY", "passive")   # see oracle/flatip_oracle.py::_load
os.environ.setdefault("GOMP_SPINCOUNT", "0")

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "czech-contriever_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

UNIT = "queries/s"
CHUNK = 1 << 18          # rows per generated corpus chunk (seeded by global chunk index)
PROBE_QUERIES = 32       # parity_probe: queries checked against an fp64 brute force per run
DUMP_BYTES = 60 << 20    # --dump-outputs payload: under 64 MB with the .npy headers

# BASELINE.json configs (SURVEY.md 8d).  bound = the roofline that applies to the scoring kernel.
WORKLOADS = {
    "c2": {"n_corpus": 1_000_000, "n_queries": 10_000, "k": 100, "store": "f32", "bound": "tensor"},
    "c3": {"n_corpus": 21_000_000, "n_queries": 100_000, "k": 100, "store": "f32", "bound": "tensor"},
    "c4": {"n_corpus": 21_000_000, "n_queries": 100_000, "k": 1000, "store": "bf16", "bound": "tensor"},
    "c5": {"n_corpus": 21_000_000, "n_queries": 64, "k": 10, "store": "f32", "bound": "hbm"},
}


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 3; 200 for --workload c5)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the last timed step's scores / ids as DIR/*.npy (see dump_outputs)")
    ap.add_argument("--impl", default="b2ip", choices=["b2ip", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--n-corpus", type=int, default=None)
    ap.add_argument("--n-queries", type=int, default=None)
    ap.add_argument("--k", type=int, default=None)
    ap.add_argument("--d", type=int, default=768)
    ap.add_argument("--store", default=None, choices=["f32", "bf16", "f16"])
    ap.add_argument("--shadow", default=None, choices=["bf16", "f16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-search-knn", action="store_true")
    ap.add_argument("--no-balance", action="store_true",
                    help="N > 1: keep equal row shards (default: shards proportional to each GPU's measured scoring rate)")
    ap.add_argument("--e2e-steps", type=int, default=5, help="timed steps of each e2e variant (<= --steps)")
    ap.add_argument("--secondary-steps", type=int, default=3)
    # CPU legs (reference arm and the cpu_baseline of the main arm)
    ap.add_argument("--ref-queries", type=int, default=0,
                    help="queries per CPU step (0: sized so that all warm-up + timed steps fit --ref-budget-s)")
    ap.add_argument("--ref-budget-s", type=float, default=180.0)
    ap.add_argument("--ref-rows", type=int, default=0,
                    help="CPU legs on the first ROWS rows only (0 = the full corpus; >0 is reported as a scaled estimate)")
    ap.add_argument("--corpus-file", default=None, help="raw float32 [n_corpus, d] file to map instead of generating")
    ap.add_argument("--extra-cpu-legs", default="", help="e.g. 'c5:1,c5:64': extra CPU timings over the same corpus")
    ap.add_argument("--cpu-baseline-queries", type=int, default=512)
    args = ap.parse_args(argv)
    w = WORKLOADS[args.workload]
    for key in ("n_corpus", "n_queries", "k", "store"):
        if getattr(args, key) is None:
            setattr(args, key, w[key])
    args.bound = w["bound"]
    if args.steps is None:
        # SURVEY 8d: latency per batch over >= 200 batches after warm-up
        args.steps = 200 if args.workload == "c5" else 3
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "measured (MEASURED_PEAKS.json)"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, \
            "fallback (B200_PROFILING.md)"


def profile_traffic(name):
    """dram bytes per launch of the dominant kernel from the committed `ncu --set full` capture:
    a constant read from profiles/, NOT measured by this run (ncu cannot run inside a bench)."""
    for cand in (name.replace("r1", "r2", 1), name):
        try:
            with open(os.path.join(ROOT, "profiles", cand)) as f:
                prof = json.load(f)
            return prof, cand
        except Exception:
            continue
    return None, None


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU every 100 ms via NVML."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            pass

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(0.1)

    def finish(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def gen_rows(torch, lo, hi, d, seed_base, device):
    """Rows [lo,hi) of the synthetic L2-normalised Gaussian matrix; chunk c (global rows
    [c*CHUNK,(c+1)*CHUNK)) always comes from seed seed_base*1000003+c, whatever the sharding."""
    for c in range(lo // CHUNK, (hi + CHUNK - 1) // CHUNK):
        c0 = c * CHUNK
        gen = torch.Generator(device=device).manual_seed(seed_base * 1000003 + c)
        x = torch.randn((CHUNK, d), generator=gen, device=device, dtype=torch.float32)
        x /= x.norm(dim=1, keepdim=True)
        a, b = max(lo, c0) - c0, min(hi, c0 + CHUNK) - c0
        yield max(lo, c0), x[a:b]


def gen_queries(torch, nq, d, device):
    gen = torch.Generator(device=device).manual_seed(4321)
    q = torch.randn((nq, d), generator=gen, device=device, dtype=torch.float32)
    q /= q.norm(dim=1, keepdim=True)
    return q


def metric_name(n_corpus, k, d):
    return f"queries/sec top-{k} exact IP search, {n_corpus / 1e6:g}M x {d}"


def workload_config(args, world, name=None, n_corpus=None, n_queries=None, k=None, store=None):
    name = name or args.workload
    n_corpus = n_corpus or args.n_corpus
    n_queries = n_queries or args.n_queries
    k = k or args.k
    store = store or args.store
    op = store if store != "f32" else (args.shadow or "bf16")
    stored = {"f32": "fp32", "bf16": "bf16-stored", "f16": "fp16-stored"}[store]
    return {
        "workload": (f"{name.upper()}: {n_corpus} x {args.d} {stored} synthetic L2-normalised corpus, "
                     f"{n_queries} queries, k={k}"),
        "n_corpus": n_corpus, "n_queries": n_queries, "k": k, "d": args.d,
        "parallelism": f"row-shard x{world} (one process per GPU; peer-direct exchange over NVLink + merge, "
                       "NCCL all-gather as fallback)",
        "l2": f"inputs exceed L2: every step streams the whole {op} operand copy of the corpus (2*d bytes/row)",
        "coarse": f"tcgen05 kind::f16 {op} operands, fp32 accumulate; fp32 rescore (fp64 accumulate)",
    }


# =============================================================================== CPU legs
def _host_corpus(args, np):
    """The synthetic corpus in host memory as float32 [rows, d] + a note saying where it came from."""
    n, d = args.n_corpus, args.d
    rows = args.ref_rows if 0 < args.ref_rows < n else n
    if args.corpus_file:
        x = np.memmap(args.corpus_file, dtype=np.float32, mode="r", shape=(n, d))
        return x[:rows], "the rows the GPU index holds (exported to host memory by the main arm)"
    try:
        import torch
        cuda = torch.cuda.is_available()
    except Exception:
        cuda = False
    x = np.empty((rows, d), dtype=np.float32)
    if cuda:
        # the generator bench.py's GPU arm uses (same seeds -> the same corpus), copied to the host
        dev = torch.device("cuda", 0)
        pin = torch.empty((CHUNK, d), dtype=torch.float32, pin_memory=True)
        for g0, r in gen_rows(torch, 0, rows, d, 1234, dev):
            m = r.shape[0]
            pin[:m].copy_(r)
            torch.cuda.synchronize()
            x[g0:g0 + m] = pin[:m].numpy()
        del pin
        torch.cuda.empty_cache()
        return x, "the same synthetic corpus as the GPU arm (torch CUDA generator, seed 1234, copied to host)"
    from concurrent.futures import ThreadPoolExecutor

    def fill(c):
        lo, hi = c * CHUNK, min(rows, (c + 1) * CHUNK)
        r = np.random.Generator(np.random.Philox(key=1234 * 1000003 + c)).standard_normal((hi - lo, d), dtype=np.float32)
        r /= np.linalg.norm(r, axis=1, keepdims=True)
        x[lo:hi] = r
    with ThreadPoolExecutor(max_workers=host_cores()) as ex:
        list(ex.map(fill, range((rows + CHUNK - 1) // CHUNK)))
    return x, "a synthetic L2-normalised Gaussian corpus of the same shape (numpy Philox; no CUDA device for the GPU arm's generator)"


def _host_queries(args, np, nq):
    try:
        import torch
        if torch.cuda.is_available():
            return gen_queries(torch, max(nq, 64), args.d, torch.device("cuda", 0))[:nq].cpu().numpy()
    except Exception:
        pass
    q = np.random.Generator(np.random.Philox(key=4321)).standard_normal((nq, args.d), dtype=np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    return q


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path -- `Indexer.search_knn`
    over `faiss.IndexFlatIP.search` (src/index.py:34-46) -- as restated in oracle/ (faiss-cpu 1.8.0
    is not installable offline; real faiss is used when importable).  Rank 0 only.  Every step
    searches `ref_queries` queries against the FULL corpus held in host memory (BASELINE.md 3);
    `value` is the measured queries/s of those steps, `ms_per_step` their measured duration."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cores = host_cores()
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm gets every host core, set BEFORE numpy /
    # OpenBLAS / libgomp are loaded
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = str(cores)
    import numpy as np
    from oracle import flatip_oracle as fo
    t_gen = time.perf_counter()
    x, corpus_note = _host_corpus(args, np)
    t_gen = time.perf_counter() - t_gen
    rows = x.shape[0]
    scale = args.n_corpus / rows
    n_pass = args.steps + args.warmup
    # calibration: a short search tells how many queries fit the time budget
    qcal = _host_queries(args, np, 256)
    cal_rows = min(rows, 1 << 17)
    fo.restatement_search(qcal[:64], x[:cal_rows], args.k)
    t0 = time.perf_counter()
    fo.restatement_search(qcal, x[:cal_rows], args.k)
    rate = 2.0 * 256 * cal_rows * args.d / (time.perf_counter() - t0)
    nq_s = args.ref_queries
    if nq_s <= 0:
        per_pass = args.ref_budget_s / max(1, n_pass)
        nq_s = int(per_pass * rate / (2.0 * rows * args.d)) // 32 * 32
        nq_s = max(32, min(2048, nq_s))
    nq_s = min(nq_s, args.n_queries)
    q = _host_queries(args, np, nq_s)
    ix = fo.make_index(x)            # faiss.IndexFlatIP(d) + add (real faiss when importable)
    ts = []
    for i in range(n_pass):
        t0 = time.perf_counter()
        ix.search(q, args.k)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            ts.append(dt)
    t = sum(ts) / len(ts)
    qps = nq_s / t / scale
    extra = []
    for leg in [s for s in args.extra_cpu_legs.split(",") if s]:
        name, b = leg.split(":")
        w, b = WORKLOADS[name], int(b)
        qb = _host_queries(args, np, b)
        t0 = time.perf_counter()
        ix.search(qb, w["k"])
        tb = time.perf_counter() - t0
        extra.append({"workload": name, "batch": b, "k": w["k"], "ms_per_batch": tb * 1e3 * scale,
                      "value": b / tb / scale, "unit": UNIT,
                      "threads_used": min(b, cores) if b < 20 else cores,
                      "note": ("faiss's sequential path (nq < 20): one thread per query" if b < 20
                               else "sgemm block path")})
    info = {
        "value": qps, "unit": UNIT, "cores": fo.num_threads(), "kind": fo.backend_kind(),
        "sample": (f"{nq_s} queries x {rows} rows ({'the FULL corpus' if rows == args.n_corpus else 'a row subset'}) "
                   f"per step, {t:.2f} s per step, k={args.k}; {corpus_note}; {fo.backend_description()}; "
                   f"host threads {cores} (OMP_NUM_THREADS/OPENBLAS_NUM_THREADS forced before load, whatever "
                   "torchrun exported)"),
        "queries_per_step": nq_s, "rows": rows, "seconds_per_step": t,
        "batch_note": ("queries per step are what fits the time budget (--ref-budget-s over warm-up + timed steps); "
                       "faiss blocks the corpus in 1,024-row sgemm calls, so a batch of ~100 queries runs the BLAS "
                       "well below its rate for >= 512 queries per step (the main arm's cpu_baseline uses 512: "
                       "~1.6x the queries/s of a 96-query step on the same cores)") if nq_s < 512 else None,
        "gflops": 2.0 * nq_s * rows * args.d / t / 1e9, "corpus_to_host_s": t_gen,
        "scaled_to": None if rows == args.n_corpus else {
            "n_corpus": args.n_corpus, "factor": scale,
            "note": "value = measured queries/s on the row subset / factor (cost is linear in rows)"},
        "extra_legs": extra,
    }
    line = {
        "impl": "reference", "metric": metric_name(args.n_corpus, args.k, args.d), "value": qps, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": info,
        "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess(args, corpus_file, extra_legs):
    """The CPU legs of the main arm run in a fresh interpreter (`--impl reference`): thread
    counts of OpenBLAS / libgomp are fixed when those libraries load, and this process has
    already loaded torch."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "0",
           "--workload", args.workload, "--n-corpus", str(args.n_corpus), "--k", str(args.k), "--d", str(args.d),
           "--ref-queries", str(min(args.cpu_baseline_queries, args.n_queries)),
           "--corpus-file", corpus_file, "--extra-cpu-legs", extra_legs]
    env = {k: v for k, v in os.environ.items()
           if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS")}
    env["CUDA_VISIBLE_DEVICES"] = ""          # the CPU legs must not touch the GPU being measured
    out = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=1500)
    if out.returncode != 0:
        return {"error": (out.stderr or out.stdout)[-400:]}
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    return line["cpu_baseline"]


# =============================================================================== GPU arm
class Dist:
    """barrier / reductions over the ranks (identity at world 1)."""

    def __init__(self, torch, dist, world, dev):
        self.torch, self.dist, self.world, self.dev = torch, dist, world, dev

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def _red(self, x, op):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max(self, x):
        return self._red(x, self.dist.ReduceOp.MAX) if self.world > 1 else x

    def sum(self, x):
        return self._red(x, self.dist.ReduceOp.SUM) if self.world > 1 else x

    def all_gather(self, x):
        """One float per rank, in rank order."""
        if self.world == 1:
            return [float(x)]
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        out = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(o.item()) for o in out]


STAT_KEYS = ("coarse_ms", "coarse_flops", "coarse_launches", "launches", "candidates", "rescored", "fallback",
             "slabs", "refresh_ms", "finalize_ms", "device_ms", "max_err_over_eps", "bound_violations")


def timed_device_steps(torch, D, index, q_dev, k, steps, warmup, world, sample_clocks_on=None, light=False):
    """W untimed + K timed searches with device-resident queries.  Returns per-step ms (max over
    ranks), the summed engine stats of the timed steps, the last result (scores, rows, (q_lo, q_hi))
    of the queries this rank owns, and the clock samples."""
    agg = {key: 0.0 for key in STAT_KEYS}

    def collect(n_steps):
        st = index.engine.stats()
        for key_a, key_s in (("coarse_ms", "coarse_ms"), ("coarse_flops", "coarse_flops"), ("coarse_launches", "coarse_launches"),
                             ("candidates", "candidates"), ("rescored", "rescored"), ("fallback", "fallback_queries"),
                             ("slabs", "slabs"), ("refresh_ms", "refresh_ms"), ("finalize_ms", "finalize_ms"),
                             ("device_ms", "total_ms"), ("bound_violations", "bound_violations")):
            agg[key_a] += st[key_s] * n_steps
        agg["launches"] += st["total_launches"] * n_steps
        agg["max_err_over_eps"] = max(agg["max_err_over_eps"], st.get("max_err_over_eps", 0.0))

    def step():
        # world > 1: the result stays partitioned over the ranks by query (rank r holds the global
        # top-k of the queries it owns) -- every query is merged once, nothing is replicated
        res = index.search_owned(q_dev, k)
        if light:                # latency regime: the counters of ONE step stand for all (fixed schedule)
            return res
        st = index.engine.stats()
        agg["coarse_ms"] += st["coarse_ms"]; agg["coarse_flops"] += st["coarse_flops"]
        agg["coarse_launches"] += st["coarse_launches"]
        # all-gather path: + the NCCL kernel and the merge kernel; the peer-direct exchange's
        # launches are already in the library's count
        agg["launches"] += st["total_launches"] + (2 if world > 1 and getattr(index, "exchange_searches", 0) == 0 else 0)
        agg["candidates"] += st["candidates"]; agg["rescored"] += st["rescored"]
        agg["fallback"] += st["fallback_queries"]; agg["slabs"] += st["slabs"]
        agg["refresh_ms"] += st["refresh_ms"]; agg["finalize_ms"] += st["finalize_ms"]
        agg["device_ms"] += st["total_ms"]
        agg["max_err_over_eps"] = max(agg["max_err_over_eps"], st.get("max_err_over_eps", 0.0))
        agg["bound_violations"] += st.get("bound_violations", 0)
        return res

    for _ in range(warmup):
        step()
    for key in agg:
        agg[key] = 0.0
    sampler = ClockSampler(sample_clocks_on) if sample_clocks_on is not None else None
    D.barrier()
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        last = step()
    e1.record()
    D.barrier()
    clocks = sampler.finish() if sampler else None
    ms = D.max(e0.elapsed_time(e1))
    if light:
        # per-kernel times of a graph-replayed search need the event nodes inside the graph: a
        # short extra pass with them enabled (3 us per node -- kept out of the timed steps above)
        index.engine.set_option("graph_timing", 1)
        for _ in range(3):
            index.search_owned(q_dev, k)
        collect(steps)
        index.engine.set_option("graph_timing", 0)
    return ms / steps, agg, last, clocks


def roofline_of(args, D, agg, steps, ms_per_step, rows_local, nq, bound, d):
    peaks, peak_src = load_peaks()
    coarse_ms = D.max(agg["coarse_ms"])
    launches = max(1, int(agg["coarse_launches"]))
    if bound == "tensor":
        achieved = agg["coarse_flops"] / (agg["coarse_ms"] / 1e3) / 1e12 if agg["coarse_ms"] > 0 else 0.0
        achieved = -D.max(-achieved)     # slowest rank
        peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
        prof, src = profile_traffic("r1_coarse_ncu.json")
        return {
            "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            "traffic": (prof["dram_bytes_read"] + prof["dram_bytes_write"]) if prof else None,
            "traffic_note": (f"CONSTANT from profiles/{src} (one `ncu --set full` capture of {prof['launch']}: "
                             f"{prof['flops']:.3e} FLOP in {prof['duration_ms']:.1f} ms), not measured by this run")
            if prof else None,
            "kernel": "coarse_filter_pair_kernel (tcgen05.mma.cta_group::2 kind::f16, fused threshold filter)",
            "peak_source": peak_src + " bf16_tflops_sustained (kernel timed inside a multi-second step)",
            "burst_peak": peaks.get("bf16_tflops"),
            "flops_per_launch_avg": agg["coarse_flops"] / launches,
            "launches": int(agg["coarse_launches"]), "kernel_ms_per_step": coarse_ms / steps,
            "kernel_share_of_step": coarse_ms / steps / ms_per_step if ms_per_step > 0 else None,
        }
    # small batches: the streaming kernel reads the 16-bit operand copy of the shard once per batch
    # -> HBM-bound.  Algorithmic bytes = rows * d * 2 (what MUST be read); SURVEY 8d's figure for an
    # fp32-stored corpus (rows * d * 4) is reported next to it.
    peak = float(peaks.get("hbm_gbs", 6650.0))
    bytes_rank = rows_local * d * 2.0 * steps
    gbs = bytes_rank / (agg["coarse_ms"] / 1e3) / 1e9 if agg["coarse_ms"] > 0 else 0.0
    gbs = -D.max(-gbs)
    prof, src = profile_traffic("r1c_stream_ncu.json")
    whole = rows_local * d * 2.0 / (ms_per_step / 1e3) / 1e9
    return {
        "bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
        "traffic": (prof["dram_bytes_read"] + prof["dram_bytes_write"]) if prof else None,
        "traffic_note": (f"CONSTANT from profiles/{src} (one `ncu --set full` capture of {prof['launch']}: "
                         f"{prof['algorithmic_bytes']:.4e} algorithmic bytes in {prof['duration_ms']:.3f} ms), "
                         "not measured by this run") if prof else None,
        "kernel": ("coarse_stream_kernel (corpus tile on the MMA's M side, resident queries, TMA-streamed 16-bit rows)"
                   if nq <= 64 else "coarse_filter_kernel<false> (TMA-streamed 16-bit corpus tiles, fused filter)"),
        "peak_source": peak_src + " hbm_gbs (copy bandwidth)",
        "bytes_per_launch_avg": bytes_rank / launches,
        "launches": int(agg["coarse_launches"]), "kernel_ms_per_step": coarse_ms / steps,
        "kernel_share_of_step": coarse_ms / steps / ms_per_step if ms_per_step > 0 else None,
        "whole_batch_gbs_16bit": whole, "whole_batch_frac_16bit": whole / peak,
        "whole_batch_gbs_fp32_bytes_survey8d": 2.0 * whole,
        "ms_per_batch": ms_per_step,
    }


def parity_probe(torch, dist, D, res, q_dev, k, d, lo, hi, world, rank, dev, rows_fn, rtol=1e-5):
    """fp64 brute force over this rank's shard for the first PROBE_QUERIES queries, all-gathered
    and merged, against the timed result: identical id sets except for ties within `rtol`
    relative of the k-th score, scores within `rtol` relative (the north_star tolerance)."""
    nqp = min(PROBE_QUERIES, q_dev.shape[0])
    qs = q_dev[:nqp].double()
    best_s = torch.full((nqp, 0), 0.0, dtype=torch.float64, device=dev)
    best_i = torch.zeros((nqp, 0), dtype=torch.int64, device=dev)
    for g0, rows in rows_fn(lo, hi):
        s = qs @ rows.double().T
        ids = torch.arange(g0, g0 + rows.shape[0], device=dev).expand(nqp, -1)
        cs, ci = torch.cat([best_s, s], dim=1), torch.cat([best_i, ids], dim=1)
        top = torch.topk(cs, min(k, cs.shape[1]), dim=1)
        best_s, best_i = top.values, torch.gather(ci, 1, top.indices)
    if best_s.shape[1] < k:       # a shard with fewer than k rows
        pad = k - best_s.shape[1]
        best_s = torch.cat([best_s, torch.full((nqp, pad), -float("inf"), dtype=torch.float64, device=dev)], 1)
        best_i = torch.cat([best_i, torch.full((nqp, pad), -1, dtype=torch.int64, device=dev)], 1)
    if world > 1:
        gs = [torch.empty_like(best_s) for _ in range(world)]
        gi = [torch.empty_like(best_i) for _ in range(world)]
        dist.all_gather(gs, best_s.contiguous())
        dist.all_gather(gi, best_i.contiguous())
        cs, ci = torch.cat(gs, 1), torch.cat(gi, 1)
        top = torch.topk(cs, k, dim=1)
        best_s, best_i = top.values, torch.gather(ci, 1, top.indices)
    Dg, Ig, (q_lo, q_hi) = res                   # this rank's queries [q_lo, q_hi) of the search
    a0, a1 = min(q_lo, nqp), min(q_hi, nqp)        # probe queries this rank holds the answer of
    ours_s, ours_i = Dg[a0 - q_lo:a1 - q_lo].double(), Ig[a0 - q_lo:a1 - q_lo]
    best_s, best_i = best_s[a0:a1], best_i[a0:a1]
    rel = ((ours_s - best_s).abs() / best_s.abs().clamp_min(1e-30)).max().item() if a1 > a0 else 0.0
    ok = rel <= rtol
    tie_swaps = 0
    bs, bi, oi = best_s.cpu(), best_i.cpu(), ours_i.cpu()
    os_ = ours_s.cpu()
    for j in range(a1 - a0):
        a, b = set(oi[j].tolist()), set(bi[j].tolist())
        if a == b:
            continue
        tie_swaps += 1
        kth = float(bs[j, -1])
        # an id on one side only must tie with the k-th score: its own score is on its side's list
        for r in a - b:
            sc = float(os_[j][oi[j] == r][0])
            ok = ok and abs(sc - kth) <= rtol * abs(kth)
        for r in b - a:
            sc = float(bs[j][bi[j] == r][0])
            ok = ok and abs(sc - kth) <= rtol * abs(kth)
    rel = D.max(rel)
    tie_swaps = int(D.sum(tie_swaps))
    ok = D.sum(0.0 if ok else 1.0) == 0.0
    return {"queries": nqp, "max_rel_score_err": rel, "queries_with_tie_swaps": tie_swaps, "rtol": rtol,
            "checked_against": "fp64 torch brute force over the full corpus (every rank's shard, all-gathered); "
                               "each rank checks the probe queries whose result it owns",
            "pass": bool(ok)}


def run_guarded(fn, torch, dist, world, group):
    """Runs one secondary workload; returns None, or what went wrong (a string) -- on EVERY rank.
    A secondary workload must not cost the primary line, so its error is recorded instead of
    raised.  N > 1: the searches are collective, so the ranks agree on the outcome over a host-side
    (gloo) group first; a rank that failed ALONE finds nobody there, times out (the group's
    timeout) and the job fails loudly instead of hanging in a half-entered NCCL collective."""
    err = None
    try:
        fn()
    except Exception as e:  # noqa: BLE001
        err = f"{type(e).__name__}: {e}"[:400]
    if world > 1:
        flag = torch.tensor([1 if err else 0], dtype=torch.int32)
        dist.all_reduce(flag, group=group)
        if int(flag.item()) and not err:
            err = "failed on another rank"
    return err


def dump_rows(np, nq, k):
    """Query rows whose answers --dump-outputs writes: all of them when their float32 scores and
    float64 ids fit DUMP_BYTES, else a fixed seeded sample (ascending), the same in every run."""
    m = min(nq, DUMP_BYTES // (12 * k + 8))
    if m == nq:
        return np.arange(nq)
    return np.sort(np.random.default_rng(0).choice(nq, m, replace=False))


def dump_outputs(out_dir, np, D_own, I_own, q_lo, nq, dist=None, group=None):
    """Writes the answer of a search of `nq` queries -- this rank holds rows [q_lo, q_lo + len(D_own))
    of it -- for the `dump_rows` queries as out_dir/query_rows.npy (float64 [m]), scores.npy
    (float32 [m,k]) and ids.npy (float64 [m,k]; exact below 2^53).  With `dist` every rank of
    `group` must call it; rank 0 gathers the slices and writes."""
    rows = dump_rows(np, nq, D_own.shape[1])
    mine = rows[(rows >= q_lo) & (rows < q_lo + D_own.shape[0])]
    part = (mine.astype(np.float64), np.asarray(D_own[mine - q_lo], dtype=np.float32),
            np.asarray(I_own[mine - q_lo], dtype=np.float64))
    if dist is not None:
        parts = [None] * dist.get_world_size(group) if dist.get_rank() == 0 else None
        dist.gather_object(part, parts, dst=0, group=group)
        if dist.get_rank() != 0:
            return
        part = tuple(np.concatenate(a) for a in zip(*parts))     # owned slices ascend with the rank
    os.makedirs(out_dir, exist_ok=True)
    for name, a in zip(("query_rows", "scores", "ids"), part):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    t_start = time.perf_counter()
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world_env == 1 and "RANK" not in os.environ:
        # convenience: relaunch under torchrun (the driver launches us that way itself)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000)] + sys.argv
        sys.exit(subprocess.call(cmd))

    import numpy as np
    import torch
    import torch.distributed as dist
    from b2ip import Engine, ShardedIndex, shard_bounds, weighted_shard_bounds
    from b2ip.indexer import Indexer

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = world_env
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b2ip needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    cpu_group = guard_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        # a host-only group for the phase where rank 0 alone drives every GPU: an NCCL barrier
        # would leave a spinning kernel on the waiting ranks' GPUs and take SMs from the measurement
        cpu_group = dist.new_group(backend="gloo")
        import datetime
        guard_group = dist.new_group(backend="gloo", timeout=datetime.timedelta(seconds=180))
    D = Dist(torch, dist, world, dev)

    N, nq, k, d = args.n_corpus, args.n_queries, args.k, args.d
    weights = None           # per-rank scoring rates (N > 1, see "balance" below); None = equal shards

    def row_shard(n_rows):
        return weighted_shard_bounds(n_rows, weights, rank) if weights else shard_bounds(n_rows, world, rank)

    lo, hi = row_shard(N)

    def build_index(store, n_rows, shadow=None):
        """Row shard [lo,hi) of the first n_rows rows of the synthetic corpus on this rank's GPU."""
        a, b = row_shard(n_rows)
        ix = ShardedIndex(d, device=local_rank, store=store)
        if shadow is not None:
            ix.engine.set_option("shadow_f16", int(shadow == "f16"))
        ix.engine.reserve(b - a)
        for g0, rows in gen_rows(torch, a, b, d, 1234, dev):
            ix.add_local(rows, g0)
        ix.engine.use_torch_stream()
        return ix, a, b

    t_ing = time.perf_counter()
    index, lo, hi = build_index(args.store, N, args.shadow)
    torch.cuda.synchronize()
    t_ing = time.perf_counter() - t_ing
    q_dev = gen_queries(torch, nq, d, dev)

    # ---------------------------------------------------------------- balance (N > 1)
    # A row-sharded search ends with its slowest rank, and under the 1 kW cap the B200s of one box
    # sustain clocks a few percent apart.  Setup, outside every timed region: a few searches on
    # equal shards measure each rank's scoring rate (FLOP / scoring-kernel time); the shards are
    # then rebuilt with sizes proportional to those rates (`weighted_shard_bounds`).
    balance = None
    if world > 1 and not args.no_balance and args.bound == "tensor":
        cal_steps = 4
        for _ in range(2):
            index.search_owned(q_dev, k)
        fl = ms = 0.0
        for _ in range(cal_steps):
            index.search_owned(q_dev, k)
            st = index.engine.stats()
            fl += st["coarse_flops"]
            ms += st["coarse_ms"]
        rates = [float(x) for x in D.all_gather(fl / max(ms, 1e-9) / 1e9)]       # TFLOP/s per rank
        spread = (max(rates) - min(rates)) / max(rates)
        balance = {"rank_tflops_equal_shards": [round(r, 1) for r in rates], "spread": round(spread, 4),
                   "applied": bool(spread > 0.005),
                   "note": "setup, untimed: shard sizes proportional to each GPU's measured scoring rate"}
        if balance["applied"]:
            weights = rates
            index.engine.close()
            del index
            torch.cuda.empty_cache()
            index, lo, hi = build_index(args.store, N, args.shadow)
            torch.cuda.synchronize()
        balance["shard_rows"] = [int(x) for x in D.all_gather(float(hi - lo))]

    # ---------------------------------------------------------------- device-resident timing
    ms_per_step, agg, last, clocks = timed_device_steps(
        torch, D, index, q_dev, k, args.steps, args.warmup, world, sample_clocks_on=local_rank,
        light=(args.bound == "hbm"))
    D_last, I_last, (own_lo, own_hi) = last
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, np, D_last.cpu().numpy(), I_last.cpu().numpy(), own_lo, nq,
                     *((dist, cpu_group) if world > 1 else ()))
    value = nq / (ms_per_step / 1e3)
    roofline = roofline_of(args, D, agg, args.steps, ms_per_step, hi - lo, nq, args.bound, d)
    def _probe_rows(a, b, ix):
        # a bf16 / fp16 store is exact w.r.t. the STORED values: the probe sees those ("same inputs")
        for g0, rows in gen_rows(torch, a, b, d, 1234, dev):
            if ix.engine.store == "bf16":
                rows = rows.bfloat16().float()
            elif ix.engine.store == "f16":
                rows = rows.half().float()
            yield g0, rows

    probe = parity_probe(torch, dist, D, last, q_dev, k, d, lo, hi, world, rank, dev,
                         lambda a, b: _probe_rows(a, b, index))
    # order-independent digest of the last step's results, summed over the ranks' query slices:
    # the id sums are identical at every N (the sharded search returns the single-GPU answer),
    # so the scaling runs check each other
    ck = torch.stack([I_last.sum(), (I_last * torch.arange(1, k + 1, device=dev)).sum()])
    sc = D_last.double().sum().reshape(1)
    if world > 1:
        dist.all_reduce(ck)
        dist.all_reduce(sc)
    checksum = {"ids_sum": int(ck[0].item()), "ids_weighted": int(ck[1].item()),
                "scores_sum_f64": float(sc.item())}
    launches = int(D.sum(agg["launches"]))

    # ---------------------------------------------------------------- end-to-end: C ABI, pageable host buffers
    e2e = None
    n_e2e = max(1, min(args.e2e_steps, args.steps))
    q_host = q_dev.cpu().numpy()                      # pageable numpy: what the reference hands over
    if not args.no_e2e:
        shm = None
        if world == 1:
            D_host = np.empty((nq, k), dtype=np.float32)
            I_host = np.empty((nq, k), dtype=np.int64)

            def step_e2e():
                index.engine.search(q_host, k, out=(D_host, I_host))   # b2ip_search(mem=HOST) via ctypes
        else:
            # one host result array shared by the ranks (POSIX shared memory): rank r downloads
            # the queries' slice it owns, rank 0 sees the whole answer
            tag = os.environ.get("MASTER_PORT", "0")
            shm = [f"/dev/shm/b2ip_bench_{tag}_{n}.bin" for n in ("D", "I")]
            if rank == 0:
                np.memmap(shm[0], dtype=np.float32, mode="w+", shape=(nq, k)).flush()
                np.memmap(shm[1], dtype=np.int64, mode="w+", shape=(nq, k)).flush()
            D.barrier()
            D_host = np.memmap(shm[0], dtype=np.float32, mode="r+", shape=(nq, k))
            I_host = np.memmap(shm[1], dtype=np.int64, mode="r+", shape=(nq, k))

            def step_e2e():
                index.search_host(q_host, k, out=(D_host, I_host))
        step_e2e()
        D.barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            step_e2e()
        D.barrier()
        ms_e = D.max((time.perf_counter() - t0) * 1e3)
        same = bool(np.array_equal(I_host[:8], I_last[:8].cpu().numpy())) if rank == 0 else None
        e2e = {"value": nq / (ms_e / n_e2e / 1e3), "unit": UNIT,
               "h2d_bytes_per_step": nq * d * 4 * world, "d2h_bytes_per_step": nq * k * 12,
               "ms_per_step": ms_e / n_e2e, "steps": n_e2e, "host_buffers": "pageable numpy (not page-locked)",
               "timing": "host wall clock around the calls, max over ranks",
               "matches_device_result": same,
               "call": ("Engine.search(numpy) -> b2ip_search_ex(mem=HOST) via ctypes" if world == 1 else
                        "ShardedIndex.search_host: every rank uploads the queries, searches, and downloads the "
                        "result slice it owns into one shared host array")}
        if shm and rank == 0:
            del D_host, I_host
            for f in shm:
                try:
                    os.unlink(f)
                except OSError:
                    pass

    # ---------------------------------------------------------------- secondary workloads
    secondary = {}

    def run_secondary(name, ix, rows_local, nq2, k2, bound, steps2, warm2, n_rows):
        q2 = q_dev[:nq2].contiguous()
        ms2, agg2, res2, clocks2 = timed_device_steps(torch, D, ix, q2, k2, steps2, warm2, world,
                                                      sample_clocks_on=local_rank, light=(bound == "hbm"))
        a, b = row_shard(n_rows)
        pr = parity_probe(torch, dist, D, res2, q2, k2, d, a, b, world, rank, dev,
                          lambda x, y: _probe_rows(x, y, ix))
        secondary[name] = {
            "metric": metric_name(n_rows, k2, d), "value": nq2 / (ms2 / 1e3), "unit": UNIT,
            "ms_per_step": ms2, "steps": steps2, "warmup": warm2, "n_queries": nq2, "k": k2,
            "store": ix.engine.store, "rows_per_gpu": rows_local,
            "roofline": roofline_of(args, D, agg2, steps2, ms2, rows_local, nq2, bound, d),
            "parity_probe": pr, "clocks": clocks2,
            "graph_replay": bool(ix.engine.stats().get("graph_mode", 0) == 2),
            "rescored_per_query": agg2["rescored"] / steps2 / nq2,
            "threshold_bootstrap_sample_rows": int(ix.engine.stats().get("sample_rows", 0)),
            "fallback_queries": int(agg2["fallback"]),
            "rank0_ms_per_step": {"coarse": agg2["coarse_ms"] / steps2, "refresh": agg2["refresh_ms"] / steps2,
                                  "finalize": agg2["finalize_ms"] / steps2, "search_device_total": agg2["device_ms"] / steps2},
        }

    def guarded(name, fn):
        err = run_guarded(fn, torch, dist, world, guard_group)
        if err:
            secondary[name] = {"error": err}

    if not args.no_secondary and args.workload == "c3":
        s2 = max(1, args.secondary_steps)
        # C5: latency regime on the same index (batch 64, k = 10), >= 200 batches
        guarded("c5_batch64_k10", lambda: run_secondary("c5_batch64_k10", index, hi - lo, 64, 10, "hbm", 200, 20, N))
        guarded("c5_batch1_k10", lambda: run_secondary("c5_batch1_k10", index, hi - lo, 1, 10, "hbm", 200, 20, N))

        # C2: 1M x 768, 10k queries (a single-GPU config: rank 0's GPU alone at N > 1 would idle
        # the others, so it is sharded like the rest and stays comparable at N = 1)
        def c2():
            ix2, a2, b2 = build_index("f32", WORKLOADS["c2"]["n_corpus"])
            try:
                run_secondary("c2_1M_10k_k100", ix2, b2 - a2, 10_000, 100, "tensor", 20, 3, WORKLOADS["c2"]["n_corpus"])
            finally:
                ix2.engine.close()

        # C4: bf16-stored corpus, k = 1000
        def c4():
            ix4, a4, b4 = build_index("bf16", N)
            try:
                run_secondary("c4_bf16_store_k1000", ix4, b4 - a4, nq, 1000, "tensor", s2, 1, N)
            finally:
                ix4.engine.close()

        guarded("c2_1M_10k_k100", c2)
        guarded("c4_bf16_store_k1000", c4)
        torch.cuda.empty_cache()

    # ---------------------------------------------------------------- CPU baseline (rank 0, N=1)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:
            avail = 1 << 62
        need = N * d * 4
        path = f"/dev/shm/b2ip_bench_corpus_{os.getpid()}.f32"
        if avail > need * 1.25 + (8 << 30):
            try:
                mm = np.memmap(path, dtype=np.float32, mode="w+", shape=(N, d))
                for r0 in range(0, N, 1 << 20):
                    m = min(1 << 20, N - r0)
                    index.engine.export_rows(r0, m, out=mm[r0:r0 + m])
                mm.flush()
                del mm
                cpu = cpu_baseline_subprocess(args, path, "c5:1,c5:64" if args.workload == "c3" else "")
            finally:
                try:
                    os.unlink(path)
                except OSError:
                    pass
        else:
            cpu = {"error": f"host memory too small for the full corpus ({avail >> 30} GiB available, {need >> 30} GiB needed)"}

    # ---------------------------------------------------------------- the drop-in call: Indexer.search_knn
    knn = None
    exchange_desc = ("peer-direct (b2ip_search_exchange)" if world > 1 and getattr(index, "exchange_searches", 0) > 0
                     else ("nccl all-gather + merge" if world > 1 else "none"))
    if not args.no_search_knn:
        q_half = q_host.astype(np.float16)            # the reference's default query dtype (model.half())
        n_knn = max(1, min(3, args.steps))

        def time_knn(ix):
            ix.search_knn(q_half[:4096], k)                                  # warm the buffers
            ts, res = [], None
            for _ in range(n_knn):
                res = None                       # the previous answer is released OUTSIDE the timed call
                t0 = time.perf_counter()         # (passage_retrieval.py:188-190 brackets search_knn alone)
                res = ix.search_knn(q_half, k)
                ts.append(time.perf_counter() - t0)
            # the drop-in's answer for the first rows == the engine's own answer for the same
            # (float16-valued) queries, ids as strings
            _, I8 = ix.index.search(q_half[:8].astype(np.float32), k)
            I8 = I8.cpu().numpy() if hasattr(I8, "cpu") else I8
            same = all([int(x) for x in res[j][0]] == I8[j].tolist() for j in range(8)) and len(res) == nq
            return min(ts), sum(ts) / len(ts), same

        if world == 1:
            # the drop-in object around the engine already in HBM
            ixr = Indexer.from_engine(index.engine, [str(i) for i in range(N)])
            best, mean, ok = time_knn(ixr)
            knn = {"value": nq / best, "unit": UNIT, "ms_per_call": best * 1e3, "ms_per_call_mean": mean * 1e3,
                   "calls": n_knn, "devices": 1, "vs_device_step": best * 1e3 / ms_per_step,
                   "queries": "pageable float16 numpy [nq,768]", "returns": "list of (list[str] * k, float32[k])",
                   "matches_engine_result": bool(ok),
                   "call": "Indexer.search_knn (b2ip/indexer.py <- reference src/index.py:34-46)"}
        else:
            # an unmodified reference driver is ONE process: it reaches the N GPUs through
            # Indexer(device="all").  The per-rank shards are dropped first, rank 0 rebuilds the
            # index through the drop-in's own index_data and times search_knn; the others wait.
            index.engine.close()
            del index
            torch.cuda.empty_cache()
            D.barrier()
            torch.cuda.synchronize()
            if rank == 0:
                ixr = Indexer(d, 0, 8, device=list(range(world)), store="f32")
                ixr.index.reserve(N)
                for g0, rows in gen_rows(torch, 0, N, d, 1234, dev):
                    ixr.index.add(rows)
                ixr.index_id_to_db_id = [str(i) for i in range(N)]
                best, mean, ok = time_knn(ixr)
                # queries per pipelined chunk (Indexer.knn_chunk): larger chunks cost the GPUs fewer
                # fixed overheads, smaller ones leave less un-overlapped id mapping at the end
                sweep = {str(ixr.knn_chunk): best * 1e3}
                for ch in (16384, 50000):
                    default_chunk, ixr.knn_chunk = ixr.knn_chunk, ch
                    sweep[str(ch)] = time_knn(ixr)[0] * 1e3
                    ixr.knn_chunk = default_chunk
                st = ixr.index.stats()
                knn = {"value": nq / best, "unit": UNIT, "ms_per_call": best * 1e3, "ms_per_call_mean": mean * 1e3,
                       "calls": n_knn, "devices": world, "vs_device_step": best * 1e3 / ms_per_step,
                       "queries": "pageable float16 numpy [nq,768]", "returns": "list of (list[str] * k, float32[k])",
                       "matches_engine_result": bool(ok),
                       "ms_per_call_by_chunk": sweep,
                       "call": "Indexer(device='all').search_knn: one process, MultiGpuEngine over all GPUs "
                               "(B2IP_DEVICES=all for an unmodified passage_retrieval.py)"}
                ixr.index.close()
            dist.barrier(group=cpu_group)       # host-side wait: the other ranks' GPUs stay idle meanwhile

    if rank == 0:
        line = {
            "metric": metric_name(N, k, d), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None,
            "dtype": f"{args.store if args.store != 'f32' else (args.shadow or 'bf16')} coarse / f32 rescore",
            "data": "synthetic", "config": workload_config(args, world),
            "e2e": e2e, "e2e_search_knn": knn, "gpu_launches": launches, "clocks": clocks, "roofline": roofline,
            "cpu_baseline": cpu, "parity_probe": probe, "result_checksum": checksum, "secondary": secondary,
            "balance": balance,
            "wall_s": round(time.perf_counter() - t_start, 1),
            "detail": {"ingest_s": t_ing, "rows_per_gpu": hi - lo,
                       "candidates_per_query_per_step": agg["candidates"] / args.steps / nq,
                       "rescored_per_query_per_step": agg["rescored"] / args.steps / nq,
                       "fallback_queries": int(agg["fallback"]), "slabs_per_step": agg["slabs"] / args.steps,
                       "max_err_over_eps": agg["max_err_over_eps"], "bound_violations": int(agg["bound_violations"]),
                       "rank0_ms_per_step": {"coarse": agg["coarse_ms"] / args.steps,
                                             "refresh": agg["refresh_ms"] / args.steps,
                                             "finalize": agg["finalize_ms"] / args.steps,
                                             "search_device_total": agg["device_ms"] / args.steps},
                       "exchange": exchange_desc},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
