"""CPU tests of the host side: the C-ABI library loads and exports every symbol include/b2ip.h
declares (no compute without a GPU -- creation must fail loudly, not fall back), the
index.faiss reader/writer, the key ordering shared by all selection kernels, and the
row-sharded search plumbing under a world_size-2 gloo group."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from helpers import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cuda_available():
    import torch
    return torch.cuda.is_available()


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    import b2ip
    return b2ip


def test_library_exports_every_declared_symbol(built):
    hdr = open(os.path.join(ROOT, "include", "b2ip.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(b2ip_[a-z_0-9]+)\s*\(", hdr))
    assert declared == set(built.SYMBOLS), declared ^ set(built.SYMBOLS)
    lib = built.load()
    for name in declared:
        assert hasattr(lib, name), name
    out = subprocess.run(["nm", "-D", "--defined-only", built.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (b2ip_[a-z_0-9]+)", out))
    assert declared <= exported


def test_bootstrap_sample_plan_invariants(built):
    """Host arithmetic of the latency regime's threshold bootstrap (csrc/b2ip_api.cu::plan_bootstrap,
    no CUDA call): swept over corpus sizes from one row to billions -- it must never fault (a zero
    grid once divided: SIGFPE on corpora of fewer than 17 tiles) and a taken sample must satisfy what
    the kernels rely on: every CTA sees a tile, only full tiles, >= 16 groups per wanted result, at
    most 1/16 of the corpus, at most `bootstrap_max_mb` of 16-bit rows."""
    import ctypes
    lib = built.load()

    def plan(n, k, cap=4096, sms=148, d_pad=768, max_mb=64):
        grid, tiles = ctypes.c_int32(-1), ctypes.c_int64(-1)
        assert lib.b2ip_debug_plan_bootstrap(n, k, cap, sms, d_pad, max_mb, ctypes.byref(grid), ctypes.byref(tiles)) == 0
        return grid.value, tiles.value

    rng = np.random.default_rng(0)
    sizes = list(range(1, 4200, 7)) + [int(x) for x in 10 ** rng.uniform(3, 10.5, 4000)] + \
        [2_625_000, 2_650_112, 21_000_000, 2 ** 31 - 1, 2 ** 32 - 1]
    taken = 0
    for n in sizes:
        k = int(rng.choice([1, 2, 10, 10, 10, 33, 42, 64, 100, 1000, 2048]))
        sms = int(rng.choice([1, 2, 16, 132, 148, 148, 160, 200]))
        d_pad = int(rng.choice([64, 128, 768, 768, 1024, 4096]))
        cap = max(4096, 4 * k)
        max_mb = int(rng.choice([0, 1, 64, 64, 1 << 20]))
        grid, tiles = plan(n, k, cap, sms, d_pad, max_mb)
        if grid == 0:
            assert tiles == 0
            continue
        taken += 1
        full_tiles = n // 128
        assert 1 <= grid <= min(sms, 160) and tiles >= grid
        assert grid * 128 >= 16 * k
        assert tiles * 16 <= (n + 127) // 128 - 1
        stride = full_tiles // tiles                       # tile t = rows [t * stride * 128, +128)
        assert stride >= 16 and (tiles - 1) * stride + 1 <= full_tiles
        assert tiles * 128 * d_pad * 2 <= max_mb << 20
        # sized for an expected list fill of cap / 6 (less a few tiles cut to a whole wave)
        assert tiles * 128 >= (6 * k * n / cap) * (1 - 1 / 8) - 128 or tiles == grid
    assert taken > 200
    # the benchmark's shapes: one GPU of eight takes the sample, a whole-corpus GPU does not
    assert plan(2_625_000, 10) == (148, 296) and plan(21_000_000, 10) == (0, 0)
    assert plan(2_625_000, 100) == (0, 0) and plan(300, 1) == (0, 0) and plan(0, 10) == (0, 0)


def test_bootstrap_group_maxima_bound_the_kth_score(built):
    """The exactness argument of the threshold bootstrap (DESIGN 4.1e), on a numpy model of the
    kernel's indexing fed by the product's own planner: tile t of the sample = rows
    [t * stride * 128, +128), group of a row = (t mod grid) * 128 + its slot in the tile.  The groups
    are disjoint, so the k-th largest group maximum can never exceed the k-th best score of the
    corpus -- for ANY scores, clustered neighbours included -- and is the sample's own k-th best
    whenever no two of its k best rows share a group."""
    import ctypes
    lib = built.load()
    rng = np.random.default_rng(5)
    for n, k, sms in [(300_000, 10, 148), (50_000, 1, 148), (9_000, 10, 148), (1_000_000, 33, 132), (123_457, 7, 16)]:
        grid, tiles = ctypes.c_int32(), ctypes.c_int64()
        lib.b2ip_debug_plan_bootstrap(n, k, 4096, sms, 768, 256, ctypes.byref(grid), ctypes.byref(tiles))
        grid, tiles = grid.value, tiles.value
        assert grid > 0
        stride = (n // 128) // tiles
        t = np.arange(tiles)
        rows = (t[:, None] * stride * 128 + np.arange(128)[None, :])             # [tiles, 128]
        groups = ((t % grid)[:, None] * 128 + np.arange(128)[None, :])
        assert rows.max() < n and len(np.unique(rows)) == rows.size
        for trial in range(3):
            scores = rng.standard_normal(n).astype(np.float32)
            if trial == 1:        # neighbouring rows score alike: runs of 16 near-equal top scores in sampled tiles
                for r0 in rows[rng.integers(0, tiles, 6), 0]:
                    scores[r0:r0 + 16] = 5.0 + 1e-3 * rng.standard_normal(16)
            if trial == 2:        # NaN scores are "empty" (ordered word 0), -inf is a real score
                scores[rows[0, :5]] = np.nan
                scores[rows[-1, 3]] = -np.inf
            gmax = np.full(grid * 128, -np.inf, dtype=np.float32)
            s_rows = np.where(np.isnan(scores[rows]), -np.inf, scores[rows])
            np.maximum.at(gmax, groups.ravel(), s_rows.ravel())
            bound = np.sort(gmax)[::-1][k - 1]
            finite = np.where(np.isnan(scores), -np.inf, scores)
            kth_corpus = np.sort(finite)[::-1][k - 1]
            kth_sample = np.sort(s_rows.ravel())[::-1][k - 1]
            assert bound <= kth_sample <= kth_corpus
            top_groups = groups.ravel()[np.argsort(s_rows.ravel())[::-1][:k]]
            if len(np.unique(top_groups)) == k:
                assert bound == kth_sample
            # the filtered slab admits every row of the exact top-k (threshold = bound - 2 eps <= bound)
            assert (finite[np.argsort(finite)[::-1][:k]] >= bound).all()


def test_library_is_sm100a_tcgen05_code(built):
    """The shipped kernels are Blackwell-native: tcgen05 MMA, TMA and TMEM loads in the SASS."""
    sass = subprocess.run(["cuobjdump", "-sass", built.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in sass, mnemonic


@pytest.mark.skipif(_cuda_available(), reason="checks the no-GPU failure mode")
def test_no_gpu_means_loud_failure_not_cpu_fallback(built):
    with pytest.raises(built.B2ipError) as ei:
        built.Engine(768, 0)
    assert "no CPU fallback" in str(ei.value)
    from src.index import Indexer
    with pytest.raises(built.B2ipError):
        Indexer(768, 0, 8)


def test_indexer_rejects_pq_without_touching_the_gpu(built):
    from src.index import Indexer
    with pytest.raises(NotImplementedError):
        Indexer(768, 16, 8)


def test_product_code_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "czech-contriever_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.lower(), os.path.join(dirpath, f)


def test_index_faiss_format_round_trip(tmp_path, built):
    from oracle import flatip_oracle as fo
    rows = synth(1000, 24, 3)
    ours, theirs = str(tmp_path / "ours.faiss"), str(tmp_path / "theirs.faiss")
    built.write_flat_ip(ours, 24, 1000, lambda r0, n: rows[r0:r0 + n])
    fo.write_index_flat_ip(theirs, rows)
    raw = open(ours, "rb").read()
    assert raw == open(theirs, "rb").read()
    assert raw[:4] == b"IxFI" and len(raw) == 45 + 4 * 1000 * 24
    d, n, blocks = built.stream_flat_ip_rows(theirs)
    assert (d, n) == (24, 1000)
    assert np.array_equal(np.concatenate(list(blocks)), rows)
    assert np.array_equal(fo.read_index_flat_ip(ours), rows)


def test_index_faiss_rejects_other_index_types(tmp_path, built):
    p = tmp_path / "pq.faiss"
    p.write_bytes(b"IxPq" + b"\0" * 64)
    with pytest.raises(NotImplementedError):
        built.stream_flat_ip_rows(str(p))
    q = tmp_path / "short.faiss"
    q.write_bytes(b"IxFI\0\0")
    with pytest.raises(ValueError):
        built.stream_flat_ip_rows(str(q))


def test_shard_bounds_partition_rows(built):
    for n in (0, 1, 7, 100, 21_000_000, 21_015_324):
        for g in (1, 2, 3, 4, 8):
            spans = [built.shard_bounds(n, g, r) for r in range(g)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            assert max(hi - lo for lo, hi in spans) <= -(-n // g)


def test_weighted_shard_bounds_partition_rows(built):
    """Speed-weighted row shards: a partition of [0, n) in rank order, sizes proportional to the
    weights up to the alignment, equal weights == equal shards, degenerate weights tolerated."""
    import b2ip
    for n in (0, 1, 1000, 21_000_000, 21_015_324):
        for w in ([1.0], [1, 1], [1.0, 0.97, 1.03, 1.0], [1300, 1340, 1290, 1335, 1310, 1352, 1301, 1322], [0, 0, 5], [0, 0]):
            g = len(w)
            spans = [b2ip.weighted_shard_bounds(n, w, r) for r in range(g)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] and a[0] <= a[1] for a, b in zip(spans, spans[1:] + [(n, n)]))
            if sum(w) > 0 and n >= 1_000_000:
                for (lo, hi), x in zip(spans, w):
                    assert abs((hi - lo) - n * x / sum(w)) <= 512
    eq = [b2ip.weighted_shard_bounds(21_000_000, [1.0] * 8, r) for r in range(8)]
    assert all(abs((hi - lo) - 2_625_000) <= 256 for lo, hi in eq)


def test_key_ordering_host_build(tmp_path):
    """keys.cuh compiled for the host: larger key <=> (higher score, then lower row); NaN -> 0."""
    src = tmp_path / "k.cu"
    src.write_text(r'''
#include <cstdio>
#include <cmath>
#include <vector>
#include "keys.cuh"
using namespace b2ip;
int main() {
    std::vector<float> v = {-INFINITY, -3.4e38f, -1.f, -1e-30f, -0.f, 0.f, 1e-30f, 0.5f, 1.f, 3.4e38f, INFINITY};
    for (size_t i = 0; i + 1 < v.size(); i++) {
        if (!(order_f32(v[i]) <= order_f32(v[i + 1]))) { printf("order %zu\n", i); return 1; }
        if (v[i] < v[i + 1] && !(make_key(v[i], 0) < make_key(v[i + 1], 4000000000u))) return 2;
        if (unorder_f32(order_f32(v[i])) != v[i]) return 3;
    }
    if (order_f32(NAN) != 0u || order_f32(-INFINITY) == 0u) return 4;
    if (!(make_key(1.f, 5) > make_key(1.f, 6))) return 5;          // tie -> lower row wins
    if (key_row(make_key(2.f, 123456789u)) != 123456789u || key_score(make_key(2.f, 1)) != 2.f) return 6;
    printf("ok\n");
    return 0;
}''')
    exe = tmp_path / "k"
    inc = os.path.join(ROOT, "czech-contriever_b200", "csrc")
    subprocess.run(["nvcc", "-O1", "-I", inc, "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0 and "ok" in out.stdout, (out.returncode, out.stdout)


# ------------------------------------------------------------------------------------------
# row-sharded search under gloo, world_size 2 (the NCCL path minus the GPU): the engine and
# the merge are replaced by CPU stand-ins built on the oracle, everything else is product code
# ------------------------------------------------------------------------------------------
_WORKER = r'''
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path[:0] = [ROOT, os.path.join(ROOT, "czech-contriever_b200"), os.path.join(ROOT, "tests")]
from oracle import flatip_oracle as fo
from b2ip.sharded import ShardedIndex
from helpers import synth

class OracleEngine:                      # CPU stand-in for b2ip.Engine (tests only)
    def __init__(self, d): self.rows = np.empty((0, d), np.float32)
    def add(self, rows): self.rows = np.concatenate([self.rows, np.asarray(rows, np.float32)])
    def search(self, q, k, mode="auto"):
        D, I = fo.search(q.numpy(), self.rows, k)
        return torch.from_numpy(D), torch.from_numpy(I)

def merge(gD, gI, k):                    # CPU stand-in for the merge kernel: score desc, row asc
    G, nq, _ = gD.shape
    D = gD.permute(1, 0, 2).reshape(nq, G * k).numpy(); I = gI.permute(1, 0, 2).reshape(nq, G * k).numpy()
    D = np.where(I >= 0, D, -np.inf)
    order = np.lexsort((np.where(I >= 0, I, 1 << 62), -D), axis=1)[:, :k]
    Dm, Im = np.take_along_axis(D, order, 1), np.take_along_axis(I, order, 1)
    Dm = np.where(Im >= 0, Dm, np.finfo(np.float32).min).astype(np.float32)
    return torch.from_numpy(Dm), torch.from_numpy(Im)

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:" + os.environ["MASTER_PORT"], rank=rank, world_size=world)
d, k = 48, 20
x, q = synth(5000, d, 1234), synth(37, d, 4321)
x[3000:3010] = x[10:20]                  # exact ties across the two shards
idx = ShardedIndex(d, engine=OracleEngine(d), merge_fn=merge)
for a, b in [(0, 900), (900, 2000), (2000, 2001), (2001, 4200), (4200, 5000)]:
    idx.add_replicated(x[a:b])           # SPMD ingest: chunk i kept by rank i % world
assert idx.ntotal_local == sum(b - a for i, (a, b) in enumerate([(0, 900), (900, 2000), (2000, 2001), (2001, 4200), (4200, 5000)]) if i % world == rank)
D, I = idx.search(torch.from_numpy(q), k)
D64, I64 = fo.brute_force_f64(q, x, k)
fo.compare_topk(D.numpy(), I.numpy(), D64.astype(np.float32), I64, q, x, rtol=1e-5)
assert np.array_equal(I.numpy(), I64), "ties must resolve to the lower GLOBAL row"
# the partitioned form: every rank holds the answer of the queries it owns
Do, Io, (qlo, qhi) = idx.search_owned(torch.from_numpy(q), k)
from b2ip.sharded import shard_bounds as sb
assert (qlo, qhi) == sb(len(q), world, rank) and np.array_equal(Io.numpy(), I64[qlo:qhi])
assert np.array_equal(Do.numpy(), D.numpy()[qlo:qhi])
# contiguous sharding through add_local + shard_bounds gives the same answer
from b2ip.sharded import shard_bounds
idx2 = ShardedIndex(d, engine=OracleEngine(d), merge_fn=merge)
lo, hi = shard_bounds(5000, world, rank)
idx2.add_local(x[lo:hi], lo)
D2, I2 = idx2.search(torch.from_numpy(q), k)
assert np.array_equal(I2.numpy(), I64)
# k larger than one shard's rows: -1 padding must survive the merge
idx3 = ShardedIndex(d, engine=OracleEngine(d), merge_fn=merge)
idx3.add_local(x[rank * 3:(rank + 1) * 3], rank * 3)
D3, I3 = idx3.search(torch.from_numpy(q[:4]), 10)
assert (np.sort(I3.numpy()[:, :6], axis=1) == np.arange(6)).all() and (I3.numpy()[:, 6:] == -1).all()
dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_sharded_search_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(f"ROOT = {ROOT!r}\n" + _WORKER)
    port = str(29000 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=port,
                   OMP_NUM_THREADS="2")
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=300)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"rank {r} ok" in o, o[-3000:]


_GUARD_WORKER = r'''
import datetime, os, sys
import torch, torch.distributed as dist
sys.path[:0] = [ROOT]
import bench
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:" + os.environ["MASTER_PORT"], rank=rank, world_size=world)
group = dist.new_group(backend="gloo", timeout=datetime.timedelta(seconds=60))
ran = []
def ok(): ran.append("ok")
def boom(): raise RuntimeError("secondary went wrong on rank %d" % rank)
def boom_on_1():
    if rank == 1: raise ValueError("only here")
assert bench.run_guarded(ok, torch, dist, world, group) is None and ran == ["ok"]
e = bench.run_guarded(boom, torch, dist, world, group)                 # every rank fails: every rank records it
assert e is not None and e.startswith("RuntimeError: secondary went wrong on rank %d" % rank), e
e = bench.run_guarded(boom_on_1, torch, dist, world, group)            # one rank fails: all of them learn it
assert (e == "failed on another rank") if rank == 0 else e.startswith("ValueError: only here"), e
assert bench.run_guarded(ok, torch, dist, world, group) is None         # and the job goes on, in step
assert bench.run_guarded(boom, torch, dist, 1, None).startswith("RuntimeError")   # world 1: no collective
dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_bench_secondary_guard_agrees_across_ranks_gloo_world2(tmp_path):
    """bench.run_guarded: a failing secondary workload is recorded, not fatal, and the ranks of a
    torchrun job take the same decision (world_size 2 over gloo; bench.py is imported without a GPU)."""
    script = tmp_path / "guard_worker.py"
    script.write_text(f"ROOT = {ROOT!r}\n" + _GUARD_WORKER)
    port = str(31000 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=port)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=300)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"rank {r} ok" in o, o[-3000:]


def test_bench_reference_arm_prints_contract_line():
    """`--impl reference` under a torchrun-like environment (OMP_NUM_THREADS=1 exported): the CPU
    arm must take every host core anyway, search the FULL (here: small) corpus, and report the
    duration of what it actually ran as ms_per_step."""
    import json
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2", LOCAL_RANK="0", CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1", "--n-corpus", "30000", "--ref-queries", "64",
                          "--extra-cpu-legs", "c5:1,c5:64"],
                         capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "queries/s" and line["value"] > 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] == len(os.sched_getaffinity(0))
    assert cb["rows"] == 30000 and cb["queries_per_step"] == 64 and cb["scaled_to"] is None
    # value and ms_per_step describe the same measured step: nothing is extrapolated
    assert abs(line["value"] - 64 / (line["ms_per_step"] / 1e3)) <= 1e-6 * line["value"]
    assert [e["batch"] for e in cb["extra_legs"]] == [1, 64]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["config"]["workload"].startswith("C3")
    # the other ranks of a torchrun launch print nothing and exit 0
    env["RANK"] = "1"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bench_steps_sets_the_timed_steps():
    """--steps is the number of timed steps however it is spelled; only its default depends on the
    workload (C5: >= 200 batches)."""
    import bench
    assert bench.parse([]).steps == 3 and bench.parse(["--workload", "c5"]).steps == 200
    for argv in (["--steps", "7"], ["--steps=7"], ["--workload", "c5", "--steps=7"], ["--workload=c5", "--steps", "7"]):
        assert bench.parse(argv).steps == 7, argv
    for argv in (["--steps", "0"], ["--warmup", "-1"]):
        with pytest.raises(SystemExit):
            bench.parse(argv)


_DUMP_WORKER = r'''
import os, sys
import numpy as np, torch.distributed as dist
sys.path[:0] = [ROOT]
import bench
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:" + os.environ["MASTER_PORT"], rank=rank, world_size=world)
rng = np.random.default_rng(1)
D = rng.standard_normal((NQ, K)).astype(np.float32)
I = rng.integers(0, 1 << 40, size=(NQ, K))
per = -(-NQ // world)
lo, hi = rank * per, min((rank + 1) * per, NQ)
bench.dump_outputs(OUT, np, D[lo:hi], I[lo:hi], lo, NQ, dist, None)
dist.destroy_process_group()
print("rank", rank, "ok")
'''


@pytest.mark.parametrize("nq,k", [(300, 10), (7000, 1000)])
def test_bench_dump_outputs_writes_the_sampled_answer(tmp_path, nq, k):
    """bench.dump_outputs: float32 scores and float64 ids (exact beyond 2^32) of every query when
    they fit, else of a fixed seeded sample under 64 MB; the same files from one process holding
    the whole answer and from two ranks each holding a slice (gathered over gloo)."""
    import bench
    rng = np.random.default_rng(1)
    D = rng.standard_normal((nq, k)).astype(np.float32)
    I = rng.integers(0, 1 << 40, size=(nq, k))
    rows = bench.dump_rows(np, nq, k)
    assert np.array_equal(rows, bench.dump_rows(np, nq, k)) and (np.diff(rows) > 0).all()
    assert (len(rows) == nq) == (nq * k * 12 <= bench.DUMP_BYTES)
    one = tmp_path / "one"
    bench.dump_outputs(str(one), np, D, I, 0, nq)
    got = {n: np.load(one / f"{n}.npy") for n in ("query_rows", "scores", "ids")}
    assert got["scores"].dtype == np.float32 and got["ids"].dtype == got["query_rows"].dtype == np.float64
    assert np.array_equal(got["query_rows"], rows) and np.array_equal(got["scores"], D[rows])
    assert np.array_equal(got["ids"].astype(np.int64), I[rows])
    assert sum(os.path.getsize(one / f"{n}.npy") for n in got) < 64_000_000
    script = tmp_path / "dump_worker.py"
    two = tmp_path / "two"
    script.write_text(f"ROOT = {ROOT!r}\nOUT = {str(two)!r}\nNQ, K = {nq}, {k}\n" + _DUMP_WORKER)
    port = str(33000 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=port)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=300)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"rank {r} ok" in o, o[-3000:]
    for n in got:
        assert (two / f"{n}.npy").read_bytes() == (one / f"{n}.npy").read_bytes(), n


class _RecordingIndex:
    """Stands in for Indexer: records the index_data call sequence."""
    def __init__(self):
        self.calls = []

    def index_data(self, ids, embeddings):
        self.calls.append((list(ids), np.array(embeddings, copy=True)))


@pytest.mark.parametrize("sizes,batch", [
    ([1500, 700, 2300], 1000), ([1000, 1000], 1000), ([5], 1000), ([999, 1, 1000, 1], 1000),
    ([300, 0, 300], 250), ([2500], 1000),
])
def test_streaming_ingest_makes_the_reference_drivers_calls(tmp_path, built, sizes, batch):
    """b2ip.ingest.index_encoded_data hands index_data the same (ids, embeddings) batches, in
    the same order, as the reference driver loop (passage_retrieval.py:65-91, restated in
    tests/helpers.py) -- without its np.vstack re-copies."""
    import pickle
    from helpers import ingest_like_reference_driver, synth
    from b2ip.ingest import index_encoded_data
    files, shards, start = [], [], 0
    for i, n in enumerate(sizes):
        emb = synth(n, 16, 100 + i, normalize=False).astype(np.float16) if n else np.zeros((0, 16), np.float16)
        ids = [str(start + j) for j in range(n)]
        start += n
        path = tmp_path / f"passages_{i:02d}"
        with open(path, "wb") as f:
            pickle.dump((ids, emb), f)
        files.append(str(path))
        shards.append((ids, emb))
    want, got = _RecordingIndex(), _RecordingIndex()
    ingest_like_reference_driver(want, [s for s in shards if len(s[0])], batch)
    index_encoded_data(got, files, batch)
    assert len(got.calls) == len(want.calls)
    for (gi, ge), (wi, we) in zip(got.calls, want.calls):
        assert gi == wi
        assert ge.dtype == we.dtype and np.array_equal(ge, we)


def test_prefetch_propagates_errors_and_order(built):
    from b2ip.ingest import prefetch
    assert list(prefetch(iter(range(50)), depth=2)) == list(range(50))

    def bad():
        yield 1
        raise KeyError("boom")
    it = prefetch(bad())
    assert next(it) == 1
    with pytest.raises(KeyError):
        next(it)


def test_dropin_launcher_replaces_src_index_in_a_reference_style_checkout(tmp_path, built):
    """`python -m b2ip.dropin script.py`: the script's own `src` package wins on sys.path (as in
    the reference checkout), yet `src.index.Indexer` is the B200 Indexer and sibling modules of
    the reference's package stay importable; the reference's faiss-importing index.py never runs."""
    import subprocess
    import sys
    co = tmp_path / "checkout"
    (co / "src").mkdir(parents=True)
    (co / "src" / "__init__.py").write_text("")
    (co / "src" / "index.py").write_text("import faiss_that_is_not_installed\n")
    (co / "src" / "other.py").write_text("VALUE = 41\n")
    # a stand-in for the (absent) beir package, shaped like the import in src/beir_utils.py:14
    dense = co / "beir" / "retrieval" / "search" / "dense"
    dense.mkdir(parents=True)
    for d in (co / "beir", co / "beir" / "retrieval", co / "beir" / "retrieval" / "search"):
        (d / "__init__.py").write_text("")
    (dense / "__init__.py").write_text("class DenseRetrievalExactSearch:\n    pass\n")
    (co / "driver.py").write_text(
        "import sys\nimport src.index\nimport src.other\n"
        "from beir.retrieval.search.dense import DenseRetrievalExactSearch as DRES\n"
        "print(src.index.Indexer.__module__, src.other.VALUE + 1, sys.argv[1:], DRES.__module__)\n"
        "try:\n    src.index.Indexer(768, 16, 8)\nexcept NotImplementedError:\n    print('pq rejected')\n")
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "czech-contriever_b200"))
    out = subprocess.run([sys.executable, "-m", "b2ip.dropin", str(co / "driver.py"), "--n_docs", "100"],
                         capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=120)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "b2ip.indexer 42 ['--n_docs', '100'] b2ip.beir_search" in out.stdout and "pq rejected" in out.stdout


def test_dropin_launcher_can_swap_a_function_the_script_defines(tmp_path, built):
    """B2IP_DEVICE_QUERIES=1: the script's own module-level `embed_queries` is replaced AFTER the
    script defined it and BEFORE its `if __name__ == "__main__":` block runs (SURVEY 8f N4)."""
    import subprocess
    import sys
    from b2ip import dropin
    script = tmp_path / "driver.py"
    script.write_text(
        "import sys\n"
        "def embed_queries(args, queries, model, tokenizer):\n    return 'host'\n"
        "def main():\n    print('embed ->', embed_queries(None, [], None, None), sys.argv[1:])\n"
        "if __name__ == '__main__':\n    main()\n")
    ns = dropin.run_script(str(script), {"embed_queries": lambda *a: "device"})
    assert ns["embed_queries"](1, 2, 3, 4) == "device"
    with pytest.raises(AttributeError):
        dropin.run_script(str(script), {"no_such_function": None})
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "czech-contriever_b200"), B2IP_DEVICE_QUERIES="1")
    # the real replacement needs torch + a model; here only that it is the one being bound
    probe = tmp_path / "probe.py"
    probe.write_text(
        "def embed_queries(args, queries, model, tokenizer):\n    return 'host'\n"
        "if __name__ == '__main__':\n    print(embed_queries.__module__, embed_queries.__name__)\n")
    out = subprocess.run([sys.executable, "-m", "b2ip.dropin", str(probe)], capture_output=True, text=True,
                         env=env, cwd=str(tmp_path), timeout=120)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "embed_queries_device" in out.stdout
    env["B2IP_DEVICE_QUERIES"] = "0"
    out = subprocess.run([sys.executable, "-m", "b2ip.dropin", str(probe)], capture_output=True, text=True,
                         env=env, cwd=str(tmp_path), timeout=120)
    assert out.stdout.split() == ["__main__", "embed_queries"]


def test_segment_map_local_to_global(built):
    """Row bookkeeping of the single-process multi-GPU engine (b2ip/multi.py)."""
    import torch
    from b2ip.multi import SegmentMap
    m = SegmentMap()
    m.append(100, 50)            # local 0..49   -> global 100..149
    assert m.single_offset() == 100
    m.append(150, 10)            # contiguous: merged into the same segment
    assert m.segments == [(0, 100, 60)] and m.single_offset() == 100
    m.append(400, 20)            # local 60..79  -> global 400..419
    m.append(1000, 5)            # local 80..84  -> global 1000..1004
    assert m.single_offset() is None and m.n_local == 85
    loc = torch.tensor([[0, 59, 60, 79], [80, 84, -1, -1]])
    assert m.to_global(loc).tolist() == [[100, 159, 400, 419], [1000, 1004, -1, -1]]
    assert list(m.overlaps(0, 100)) == []
    assert list(m.overlaps(120, 405)) == [(20, 120, 40), (60, 400, 5)]
    assert list(m.overlaps(419, 2000)) == [(79, 419, 1), (80, 1000, 5)]
    with pytest.raises(ValueError):
        m.append(900, 1)


def test_multi_engine_levels_its_shards(built):
    """MultiGpuEngine.add cuts every chunk so the shards' totals stay level (ADVICE r1: the
    remainder used to go to the lowest-numbered devices), whatever the chunk sizes."""
    import random
    from b2ip.multi import level_split
    rnd = random.Random(3)
    for _ in range(3000):
        G = rnd.randint(1, 8)
        tot = [0] * G
        for _ in range(rnd.randint(1, 12)):
            n = rnd.choice([0, 1, 2, G - 1, G, G + 1, rnd.randint(0, 50)])
            take = level_split(tot, n)
            assert sum(take) == n and min(take) >= 0
            tot = [a + b for a, b in zip(tot, take)]
            assert max(tot) - min(tot) <= 1, tot
    assert level_split([0, 0, 0, 0], 3) in ([1, 1, 1, 0], [0, 1, 1, 1], [1, 0, 1, 1], [1, 1, 0, 1])
    assert level_split([3, 2, 2], 1) == [0, 1, 0]


class _OracleBackedEngine:
    """CPU stand-in for b2ip.Engine in the Indexer host-logic test (tests only): keeps the rows
    in the storage type it was created with and answers searches with the oracle."""
    created = []

    def __init__(self, d, device=0, store="f32", shadow=None):
        self.d, self.device, self.store = d, device, store
        self.rows = np.empty((0, d), np.float32)
        _OracleBackedEngine.created.append(store)

    def reserve(self, n): pass
    def close(self): pass

    @property
    def ntotal(self): return self.rows.shape[0]

    def add(self, rows):
        rows = np.asarray(rows)
        if self.store == "f16":
            rows = rows.astype(np.float16)
        self.rows = np.concatenate([self.rows, rows.astype(np.float32)])

    def export_rows(self, r0, n): return self.rows[r0:r0 + n].copy()

    def search(self, q, k, mode="auto", out=None):
        from oracle import flatip_oracle as fo
        return fo.search(np.asarray(q, np.float32), self.rows, k)


def test_indexer_host_logic_with_a_stand_in_engine(tmp_path, built, monkeypatch):
    """The drop-in Indexer above the C ABI, on CPU: same calls as the reference restatement
    (oracle.OracleIndexer <- reference src/index.py:15-73) give the same ids, scores, files and
    the reference's `index_id_to_db_id[-1]` quirk; float16 chunks select the lossless fp16 store and
    a later fp32 chunk migrates the rows to fp32 master storage."""
    from oracle import flatip_oracle as fo
    from helpers import synth
    import b2ip.indexer as bi
    monkeypatch.setattr(bi, "Engine", _OracleBackedEngine)
    _OracleBackedEngine.created.clear()
    d = 32
    a = (synth(300, d, 1, normalize=False)).astype(np.float16)
    b = (synth(200, d, 2, normalize=False)).astype(np.float16)
    c = synth(100, d, 3, normalize=False)                       # fp32, not fp16-valued
    ours, ref = bi.Indexer(d, 0, 8, device=0), fo.OracleIndexer(d, 0, 8)
    for idx in (ours, ref):
        idx.index_data([f"p{i}" for i in range(300)], a)
        idx.index_data([f"p{300 + i}" for i in range(200)], b)
    assert ours.index.store == "f16" and _OracleBackedEngine.created == ["f32", "f16"]
    q = synth(7, d, 4, normalize=False).astype(np.float16)
    for (gi, gs), (wi, ws) in zip(ours.search_knn(q, 10), ref.search_knn(q, 10)):
        assert gi == wi and isinstance(gi[0], str) and np.array_equal(gs, ws) and gs.dtype == np.float32
    for idx in (ours, ref):
        idx.index_data([f"p{500 + i}" for i in range(100)], c)
    assert ours.index.store == "f32" and ours.index.ntotal == 600          # migrated, nothing lost
    assert np.array_equal(ours.index.rows, ref.rows)
    got, want = ours.search_knn(q, 10), ref.search_knn(q, 10)
    for (gi, gs), (wi, ws) in zip(got, want):
        assert gi == wi and np.array_equal(gs, ws)
    # persistence: byte-identical index.faiss, same meta, and a reload answers the same
    da, db = tmp_path / "a", tmp_path / "b"
    da.mkdir(); db.mkdir()
    ours.serialize(str(da)); ref.serialize(str(db))
    assert (da / "index.faiss").read_bytes() == (db / "index.faiss").read_bytes()
    assert (da / "index_meta.faiss").read_bytes() == (db / "index_meta.faiss").read_bytes()
    again = bi.Indexer(d, 0, 8, device=0)
    again.deserialize_from(str(db))
    for (gi, gs), (wi, ws) in zip(again.search_knn(q, 10), want):
        assert gi == wi and np.array_equal(gs, ws)
    # fewer rows than k: faiss pads with -1 and the reference maps -1 to the LAST id (src/index.py:44)
    small, small_ref = bi.Indexer(d, 0, 8, device=0), fo.OracleIndexer(d, 0, 8)
    for idx in (small, small_ref):
        idx.index_data(["x", "y", "z"], c[:3])
    (gi, gs), (wi, ws) = small.search_knn(q[:1], 5)[0], small_ref.search_knn(q[:1], 5)[0]
    assert gi == wi and gi[3:] == ["z", "z"] and np.array_equal(gs, ws)
    assert small.search_knn(np.zeros((0, d), np.float32), 5) == []
    with pytest.raises(NotImplementedError):
        bi.Indexer(d, 8, 8)


def test_hostmap_builds_the_reference_result_objects(built):
    """csrc/hostmap.c against the reference comprehension it replaces (src/index.py:44-45):
    same strings (identity for exact `str` ids, `str(x)` otherwise), negative rows index from
    the end like a Python list, out-of-range rows raise IndexError, score rows are passed through."""
    hm = built.load_hostmap()
    rng = np.random.default_rng(5)
    for ids in ([f"doc{i}" for i in range(1000)], list(range(1000)), [f"d{i}" if i % 2 else i for i in range(1000)]):
        I = rng.integers(-3, 1000, size=(37, 11), dtype=np.int64)
        D = rng.random((37, 11), dtype=np.float32)
        want = [([str(ids[i]) for i in row], D[j]) for j, row in enumerate(I)]
        got = hm.map_ids(ids, I, 37, 11, list(D))
        assert len(got) == 37 and all(isinstance(t, tuple) and len(t) == 2 for t in got)
        assert [g[0] for g in got] == [w[0] for w in want]
        assert all(type(x) is str for g in got for x in g[0])
        assert all(np.array_equal(g[1], w[1]) and g[1].base is D for g, w in zip(got, want))
        if isinstance(ids[int(I[0, 0])], str):
            assert got[0][0][0] is ids[int(I[0, 0])]                 # no copy of an exact str
        assert hm.map_ids(ids, I, 37, 11, None) == [w[0] for w in want]
    with pytest.raises(IndexError):
        hm.map_ids(["a", "b"], np.array([[0, 2]], dtype=np.int64), 1, 2, None)
    with pytest.raises(IndexError):
        hm.map_ids([], np.array([[-1]], dtype=np.int64), 1, 1, None)          # reference: [][-1]
    with pytest.raises(ValueError):
        hm.map_ids(["a"], np.zeros((2, 2), dtype=np.int32), 2, 2, None)       # not int64[nq*k]
    assert hm.map_ids(["a"], np.zeros((0, 4), dtype=np.int64), 0, 4, []) == []


def test_hostmap_keeps_the_garbage_collector_out_of_the_way(built):
    """map_ids switches the cyclic collector off while it allocates its 2*nq containers (every
    full collection would walk the whole id list) and puts it back as it found it, also on the
    error path; list[str] rows and (list[str], ndarray) tuples leave the collector's lists, rows
    that hold anything else than exact `str` ids stay tracked."""
    import gc
    hm = built.load_hostmap()
    ids = [f"doc{i}" for i in range(50)]
    I = np.arange(12, dtype=np.int64).reshape(3, 4)
    D = np.zeros((3, 4), np.float32)
    was = gc.isenabled()
    try:
        for state in (True, False):
            gc.enable() if state else gc.disable()
            got = hm.map_ids(ids, I, 3, 4, list(D))
            assert gc.isenabled() == state
            assert not any(gc.is_tracked(t) or gc.is_tracked(t[0]) for t in got)
            with pytest.raises(IndexError):
                hm.map_ids(ids, I + 48, 3, 4, list(D))
            assert gc.isenabled() == state
        got = hm.map_ids(ids, I, 3, 4, [[0.0]] * 3)                  # tracked score rows: tuples stay tracked
        assert all(gc.is_tracked(t) and not gc.is_tracked(t[0]) for t in got)
        got = hm.map_ids(list(range(50)), I, 3, 4, None)             # str(id) path: rows stay tracked
        assert all(gc.is_tracked(r) for r in got)
    finally:
        gc.enable() if was else gc.disable()


def test_search_knn_chunk_pipeline_equals_one_search(built, monkeypatch):
    """search_knn searches in chunks on a background thread and maps ids chunk by chunk: any
    chunk size gives the result of one whole search, for numpy and (CPU) torch queries."""
    import torch
    from oracle import flatip_oracle as fo
    import b2ip.indexer as bi
    monkeypatch.setattr(bi, "Engine", _OracleBackedEngine)
    d = 16
    x, q = synth(400, d, 11), synth(23, d, 12)
    ours, ref = bi.Indexer(d, 0, 8, device=0, store="f32"), fo.OracleIndexer(d, 0, 8)
    for idx in (ours, ref):
        idx.index_data([f"p{i}" for i in range(400)], x)
    want = ref.search_knn(q, 9)
    for chunk in (1, 5, 23, 1000):
        ours.knn_chunk = chunk
        for qq in (q, q.astype(np.float64), torch.from_numpy(q)):
            got = ours.search_knn(qq, 9)
            assert len(got) == 23
            for (gi, gs), (wi, ws) in zip(got, want):
                # (the stand-in engine's BLAS blocking depends on the chunk size: last-bit noise)
                assert gi == wi and np.allclose(gs, ws, rtol=1e-6, atol=0) and gs.dtype == np.float32


def test_iter_batches_properties(built):
    """Property test of the streaming ingest's batcher over random shard sizes: the batches
    concatenate back to the shards in order, every batch but the last has exactly `batch` rows,
    ids stay aligned with rows, and batches inside one shard are zero-copy views."""
    from hypothesis import given, settings, strategies as st
    from b2ip.ingest import iter_batches

    @settings(max_examples=60, deadline=None)
    @given(st.lists(st.integers(min_value=0, max_value=40), min_size=0, max_size=8),
           st.integers(min_value=1, max_value=25))
    def check(sizes, batch):
        shards, start = [], 0
        for n in sizes:
            emb = np.arange(start, start + n, dtype=np.float32)[:, None] * np.ones((1, 3), np.float32)
            shards.append(([f"id{start + j}" for j in range(n)], emb))
            start += n
        out = list(iter_batches(iter(shards), batch))
        total = sum(sizes)
        assert sum(len(ids) for ids, _ in out) == total
        if total:
            assert all(len(ids) == batch for ids, _ in out[:-1]) and 1 <= len(out[-1][0]) <= batch
            assert [i for ids, _ in out for i in ids] == [f"id{j}" for j in range(total)]
            rows = np.concatenate([e for _, e in out])
            assert np.array_equal(rows[:, 0], np.arange(total, dtype=np.float32))
            for ids, e in out:
                assert len(ids) == e.shape[0]
        else:
            assert out == []
    check()
    big = (list(range(10)), np.zeros((10, 4), np.float32))
    (_, first), (_, second) = list(iter_batches([big], 5))
    assert first.base is big[1] and second.base is big[1]        # views, not copies


def test_header_is_plain_c_and_declares_what_the_binding_lists(built):
    """include/b2ip.h is the drop-in boundary: it must compile as C99 (no C++ in the ABI) and
    declare exactly the functions the ctypes binding lists (b2ip.SYMBOLS)."""
    import re
    import subprocess
    hdr = os.path.join(ROOT, "include", "b2ip.h")
    out = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-fsyntax-only", "-x", "c", hdr],
                         capture_output=True, text=True)
    assert out.returncode == 0 and not out.stderr.strip(), out.stderr
    text = re.sub(r"/\*.*?\*/", "", open(hdr).read(), flags=re.S)
    declared = set(re.findall(r"\b(b2ip_[a-z0-9_]+)\s*\(", text))
    assert declared == set(built.SYMBOLS), declared ^ set(built.SYMBOLS)
