"""bench.py --dump-outputs on the GPU: what the timed path computed in its last step, written so that
two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs_repeat_and_are_the_exact_top_k(tmp_path):
    """Two runs with the same arguments write identical arrays, and they are the exact top-k of the
    benchmark's own seeded corpus and queries (checked against the CPU oracle on a subset).
    6000 queries at k = 1000 do not fit the dump: a sample is written."""
    import torch
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import bench
    from oracle import flatip_oracle as fo
    n, nq, k, d = 60_000, 6000, 1000, 768
    argv = ["--n-corpus", str(n), "--n-queries", str(nq), "--k", str(k), "--steps", "2", "--warmup", "1",
            "--no-e2e", "--no-secondary", "--no-cpu-baseline", "--no-search-knn"]
    runs = []
    for i in range(2):
        out_dir = tmp_path / f"run{i}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv, "--dump-outputs", str(out_dir)],
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-3000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2 and line["parity_probe"]["pass"]
        runs.append({name: np.load(out_dir / f"{name}.npy") for name in ("query_rows", "scores", "ids")})
    a, b = runs
    for name in a:
        assert np.array_equal(a[name], b[name]), name
    rows = a["query_rows"].astype(np.int64)
    assert np.array_equal(rows, bench.dump_rows(np, nq, k)) and len(rows) < nq
    assert a["scores"].shape == a["ids"].shape == (len(rows), k)
    dev = torch.device("cuda", 0)
    x = torch.cat([r for _, r in bench.gen_rows(torch, 0, n, d, 1234, dev)]).cpu().numpy()
    q = bench.gen_queries(torch, nq, d, dev).cpu().numpy()
    sub = np.arange(0, len(rows), 41)
    Do, Io = fo.search(q[rows[sub]], x, k)
    fo.compare_topk(a["scores"][sub], a["ids"][sub].astype(np.int64), Do, Io, q[rows[sub]], x, rtol=1e-5)
