"""GPU parity tests: the CUDA path, called through the C ABI (ctypes -> libb2ip.so), against
the CPU oracle (oracle/flatip_oracle.c) on the same seeded inputs.

Acceptance (BASELINE.json north_star): identical top-k index sets, differences only among
ties whose scores are within 1e-5 relative; scores within 1e-5 relative
(oracle.flatip_oracle.compare_topk, rtol = 1e-5)."""
import os
import pickle

import numpy as np
import pytest

from helpers import ingest_like_reference_driver, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

RTOL = 1e-5


@pytest.fixture(scope="module")
def fo():
    from oracle import flatip_oracle
    return flatip_oracle


def _engine(x, device=0, store="f32"):
    from b2ip import Engine
    e = Engine(x.shape[1], device, store=store)
    e.add(x)
    return e


def test_library_reports_sm100():
    import b2ip
    assert b"sm_100a" in b2ip.load().b2ip_version()


def test_coarse_scores_match_bf16_matmul():
    """The tcgen05 mainloop alone: raw scores vs torch on the same bf16-rounded operands."""
    import torch
    x = synth(1000, 768, 1234)
    q = synth(200, 768, 4321)
    e = _engine(x)
    qt = torch.from_numpy(q).cuda()
    got = e.debug_coarse_scores(qt, 0, 1000).cpu().numpy()
    xr = torch.from_numpy(x).cuda().bfloat16().float()
    qr = qt.bfloat16().float()
    want = (qr.double() @ xr.double().T).float().cpu().numpy()
    # products of bf16 values are exact in fp32; only the accumulation order differs
    np.testing.assert_allclose(got, want, rtol=0, atol=2e-5)
    # second call at a row offset (multiple of the 256-row tile)
    got2 = e.debug_coarse_scores(qt, 512, 488).cpu().numpy()
    np.testing.assert_allclose(got2, want[:, 512:], rtol=0, atol=2e-5)


@pytest.mark.parametrize("mode", ["tensor", "exact"])
@pytest.mark.parametrize("n,nq,k,d", [
    (5000, 64, 100, 768),
    (20000, 300, 10, 768),
    (3000, 33, 1, 64),
    (4097, 129, 99, 128),
    (10000, 17, 101, 768),
    (30000, 50, 1000, 256),
    (257, 5, 100, 768),
])
def test_search_matches_oracle(fo, mode, n, nq, k, d):
    x = synth(n, d, 1234)
    q = synth(nq, d, 4321)
    e = _engine(x)
    D, I = e.search(q, k, mode=mode)
    Do, Io = fo.search(q, x, k)
    assert D.dtype == np.float32 and I.dtype == np.int64
    assert (np.diff(D, axis=1) <= 0).all(), "rows must be score-descending"
    fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)
    st = e.stats()
    assert st["nq"] == nq and st["ntotal"] == n
    if mode == "tensor":
        assert st["coarse_launches"] >= 1 and st["fallback_queries"] == 0


@pytest.mark.parametrize("nq", [1, 2, 16, 64, 128, 129, 2048])
@pytest.mark.parametrize("k", [10, 100])
def test_small_query_batches_latency_regime(fo, nq, k):
    """BASELINE config 5 regime: batches of 1-64 queries (fixed, sync-free slab schedule up to
    2048 queries) over a corpus that spans several slabs."""
    x = synth(200_000, 768, 1234)
    q = synth(nq, 768, 4321)
    e = _engine(x)
    D, I = e.search(q, k)
    st = e.stats()
    assert st["slabs"] >= 2 and st["fallback_queries"] == 0
    Do, Io = fo.search(q, x, k)
    fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)


@pytest.mark.parametrize("nq,k,d,store", [(1, 10, 768, "f32"), (7, 10, 768, "f32"), (33, 100, 128, "f32"),
                                          (64, 10, 768, "f32"), (64, 100, 896, "f32"), (48, 10, 768, "f16"),
                                          (64, 1000, 256, "bf16")])
def test_geometric_slab_schedule_small_batches(fo, nq, k, d, store):
    """Batches of <= 64 queries with the threshold bootstrap off (option bootstrap=0) run the
    geometric slab schedule: one coarse launch per slab, a threshold refresh between slabs, at
    least three slabs over this corpus.  The answer must be the oracle's on the stored
    values, and the same launch sequence replayed from a CUDA graph must reproduce it bit for bit,
    with the same candidate counts and rescored rows."""
    x = synth(300_000, d, 99)
    q = synth(nq, d, 100)
    e = _engine(x, store=store)
    e.set_option("graph", 0)
    e.set_option("bootstrap", 0)
    D0, I0 = e.search(q, k)
    s0 = e.stats()
    assert s0["coarse_launches"] == s0["slabs"] >= 3 and s0["fallback_queries"] == 0
    assert s0["graph_mode"] == 0 and s0["sample_rows"] == 0
    xs = e.export_rows(0, x.shape[0]) if store != "f32" else x       # the values actually stored
    Do, Io = fo.search(q, xs, k)
    fo.compare_topk(D0, I0, Do, Io, q, xs, rtol=RTOL)
    # captured once, then replayed three times
    e.set_option("graph", 1)
    for it in range(4):
        Dg, Ig = e.search(q, k)
        sg = e.stats()
        assert sg["graph_mode"] == (1 if it == 0 else 2)
        assert np.array_equal(Ig, I0) and np.array_equal(Dg, D0)
        assert sg["candidates"] == s0["candidates"] and sg["rescored"] == s0["rescored"]
        assert sg["coarse_launches"] == sg["slabs"] == s0["slabs"] and sg["fallback_queries"] == 0


def test_small_batches_replay_a_cuda_graph(fo):
    """The fixed launch sequence of a small batch is captured once per shape and replayed: the
    replays must pick up NEW query / output buffers (DynArgs) and give the oracle's answer, for
    host and device buffers, and per-kernel timings must survive inside the graph."""
    import torch
    x = synth(150_000, 768, 77)
    e = _engine(x)
    modes = []
    for it in range(5):
        q = synth(48, 768, 1000 + it)                      # new queries, new buffers every call
        D, I = e.search(q, 10)
        st = e.stats()
        modes.append(st["graph_mode"])
        assert st["fallback_queries"] == 0 and st["slabs"] >= 2 and st["coarse_launches"] == st["slabs"]
        Do, Io = fo.search(q, x, 10)
        fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)
        assert st["total_ms"] > 0
    assert modes[0] == 1 and set(modes[1:]) == {2}, modes
    # per-kernel times inside a graph are opt-in (event-record nodes cost ~3 us each)
    assert e.stats()["coarse_ms"] == 0
    e.set_option("graph_timing", 1)
    for it in range(2):
        e.search(q, 10)
        st = e.stats()
        assert st["graph_mode"] == it + 1
    assert 0 < st["coarse_ms"] <= st["total_ms"] and st["finalize_ms"] > 0
    e.set_option("graph_timing", 0)
    qd = torch.from_numpy(synth(48, 768, 5)).cuda()
    outs = []
    for it in range(3):                                   # device buffers: fresh output tensors per call
        Dd, Id = e.search(qd, 10)
        outs.append((Dd, Id))
    assert all(torch.equal(o[1], outs[0][1]) and torch.equal(o[0], outs[0][0]) for o in outs)
    Do, Io = fo.search(qd.cpu().numpy(), x, 10)
    fo.compare_topk(outs[2][0].cpu().numpy(), outs[2][1].cpu().numpy(), Do, Io, qd.cpu().numpy(), x, rtol=RTOL)
    # rows added after a capture: the old graph must not be replayed for the new corpus size
    e.add(synth(1000, 768, 78))
    x2 = np.concatenate([x, synth(1000, 768, 78)])
    q = synth(48, 768, 2000)
    D, I = e.search(q, 10)
    assert e.stats()["graph_mode"] == 1
    Do, Io = fo.search(q, x2, 10)
    fo.compare_topk(D, I, Do, Io, q, x2, rtol=RTOL)
    # graph off: same answer from plain launches
    e.set_option("graph", 0)
    D0, I0 = e.search(q, 10)
    assert e.stats()["graph_mode"] == 0 and np.array_equal(I0, I) and np.array_equal(D0, D)


@pytest.mark.parametrize("nq,k,d,store,n", [(1, 10, 768, "f32", 300_000), (7, 1, 768, "f32", 300_000),
                                            (33, 40, 128, "f32", 300_000), (64, 10, 768, "f32", 400_000),
                                            (64, 20, 896, "f32", 150_000), (48, 10, 768, "f16", 300_000),
                                            (64, 33, 256, "bf16", 300_000), (20, 10, 768, "f32", 9_000)])
def test_threshold_bootstrap_equals_the_geometric_schedule(fo, nq, k, d, store, n):
    """Batches of <= 64 queries take their first threshold from ONE group-max launch over a sample
    of the corpus (coarse_stream_kernel<NQ, true> + bootstrap_threshold_kernel) followed by one
    filtered slab over all rows, instead of the geometric slab schedule (option bootstrap=0).  The
    threshold only decides which rows are listed; the answer is the exact top-k either way: bit
    for bit the same ids and scores, and the oracle's."""
    x = synth(n, d, 501)
    # neighbouring rows that score alike (consecutive passages of one article): runs of 24 near-copies
    # of one row, right where the sample's first tiles lie and elsewhere
    rng = np.random.default_rng(7)
    for r0 in (0, 64, 4096, n // 2, n - 4000):
        x[r0:r0 + 24] = x[r0] + 1e-3 * rng.standard_normal((24, d)).astype(np.float32)
    q = synth(nq, d, 502)
    q[0] = x[5]                                       # a query whose best rows ARE such a run
    e = _engine(x, store=store)
    e.set_option("graph", 0)
    Db, Ib = e.search(q, k)
    sb = e.stats()
    e.set_option("bootstrap", 0)
    Dg, Ig = e.search(q, k)
    sg = e.stats()
    assert sb["slabs"] == 2 and sb["coarse_launches"] == 2 and sb["sample_rows"] >= 16 * k    # sample + one filtered slab
    assert sb["sample_rows"] <= n // 16 and sg["sample_rows"] == 0 and sg["slabs"] >= 2
    assert sb["fallback_queries"] == 0 and sg["fallback_queries"] == 0
    assert sb["bound_violations"] == 0 and sb["max_err_over_eps"] < 1.0
    assert np.array_equal(Ib, Ig) and np.array_equal(Db, Dg)
    # lists stay well inside their capacity
    assert sb["candidates"] / nq < 0.5 * max(4096, 4 * k)
    xs = e.export_rows(0, n) if store != "f32" else x
    Do, Io = fo.search(q, xs, k)
    fo.compare_topk(Db, Ib, Do, Io, q, xs, rtol=RTOL)
    # replayed from a CUDA graph, with new queries each time
    e.set_option("bootstrap", 1)
    e.set_option("graph", 1)
    for it in range(3):
        q2 = synth(nq, d, 600 + it)
        D2, I2 = e.search(q2, k)
        assert e.stats()["graph_mode"] == (1 if it == 0 else 2) and e.stats()["sample_rows"] == sb["sample_rows"]
        Do, Io = fo.search(q2, xs, k)
        fo.compare_topk(D2, I2, Do, Io, q2, xs, rtol=RTOL)


def test_large_k_small_batches_keep_the_geometric_schedule(fo):
    """The sample would be more than 1/16 of the corpus for k > ~42 (at the default list capacity;
    the limit is soft: a sample a few tiles past a whole wave is cut to the wave): those batches
    keep the geometric slab schedule."""
    x = synth(300_000, 256, 11)
    q = synth(16, 256, 12)
    e = _engine(x)
    for k, boot in ((42, True), (60, False), (100, False), (1000, False)):
        D, I = e.search(q, k)
        st = e.stats()
        assert (st["sample_rows"] > 0) == boot and st["fallback_queries"] == 0, (k, st)
        Do, Io = fo.search(q, x, k)
        fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)


def test_threshold_bootstrap_with_unusable_samples(fo):
    """Degenerate samples -> the search must still be exact (through the exact path if a list
    overflows): (a) rows in ascending score order; (b) NaN / inf rows inside the sampled tiles;
    (c) a corpus of copies of one row (every group maximum ties, every row is admitted)."""
    d, n, k = 256, 200_000, 10
    base = synth(1, d, 1)[0]
    # (a) every row a positive multiple of one direction, ascending with the row number
    x = np.outer(np.linspace(0.1, 1.0, n, dtype=np.float32), base).astype(np.float32)
    q = np.stack([base, 0.5 * base]).astype(np.float32)
    e = _engine(x)
    D, I = e.search(q, k)
    st = e.stats()
    Do, Io = fo.search(q, x, k)
    fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)
    assert st["sample_rows"] > 0
    # (b) non-finite rows in the first tiles (always sampled) and around the corpus
    x = synth(n, d, 2)
    x[3, 0] = np.nan
    x[40, 5] = np.inf
    x[100_000, 7] = -np.inf
    x[1000:1010] = 0.0
    q = synth(9, d, 3)
    e = _engine(x)
    D, I = e.search(q, k)
    Do, Io = fo.search(q, x, k)
    fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)
    # (c) all rows identical: every score ties, faiss keeps the k lowest rows
    x = np.repeat(synth(1, d, 4), n, axis=0)
    q = synth(3, d, 5)
    e = _engine(x)
    D, I = e.search(q, k)
    Do, Io = fo.search(q, x, k)
    fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)
    assert np.array_equal(I, np.tile(np.arange(k), (3, 1)))


@pytest.mark.parametrize("nq", [8, 3000])
def test_ascending_scores_overflow_every_list(fo, nq):
    """Adversarial order: rows sorted by increasing score, every row beats the running threshold,
    the candidate lists overflow (in both slab schedules) and the exact path takes over."""
    u = synth(1, 128, 3)[0]
    n = 60_000
    x = (u[None, :] * (1.0 + np.arange(n, dtype=np.float32)[:, None] * 1e-5)).astype(np.float32)
    q = np.tile(u[None, :], (nq, 1)) * np.linspace(0.5, 1.5, nq, dtype=np.float32)[:, None]
    e = _engine(x)
    D, I = e.search(q, 100)
    assert e.stats()["fallback_queries"] > 0
    Do, Io = fo.search(q, x, 100)
    fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)
    assert np.array_equal(I[0], np.arange(n - 1, n - 101, -1))


def test_c1_full_config(fo):
    """BASELINE config 1 in full: 100k x 768 corpus, 1k queries, k=100."""
    x = synth(100_000, 768, 1234)
    q = synth(1000, 768, 4321)
    e = _engine(x)
    D, I = e.search(q, 100)
    Do, Io = fo.search(q, x, 100)
    r = fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)
    assert r["queries"] == 1000


@pytest.mark.parametrize("mode", ["tensor", "exact"])
def test_fewer_rows_than_k_pads_like_faiss(fo, mode):
    x = synth(37, 768, 1)
    q = synth(9, 768, 2)
    e = _engine(x)
    D, I = e.search(q, 100, mode=mode)
    Do, Io = fo.search(q, x, 100)
    assert (I[:, 37:] == -1).all() and (D[:, 37:] == np.finfo(np.float32).min).all()
    fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)


def test_empty_index_and_empty_queries():
    from b2ip import Engine
    e = Engine(768, 0)
    D, I = e.search(synth(3, 768, 0), 10)
    assert (I == -1).all() and (D == np.finfo(np.float32).min).all()
    e.add(synth(100, 768, 1))
    D, I = e.search(np.zeros((0, 768), np.float32), 10)
    assert D.shape == (0, 10) and I.shape == (0, 10)


@pytest.mark.parametrize("mode", ["tensor", "exact"])
def test_duplicate_rows_keep_lower_row(fo, mode):
    """Exact ties: faiss's strict insertion keeps the earlier (lower) row at the boundary."""
    base = synth(40, 128, 7)
    x = np.tile(base, (20, 1))            # every row appears 20 times
    q = synth(12, 128, 8)
    e = _engine(x)
    D, I = e.search(q, 50, mode=mode)
    D64, I64 = fo.brute_force_f64(q, x, 50)   # stable: score desc, row asc
    fo.compare_topk(D, I, D64.astype(np.float32), I64, q, x, rtol=RTOL)
    # among equal scores our order is row-ascending and the k-th boundary keeps lower rows
    assert np.array_equal(I, I64)


def test_identity_corpus_known_answer():
    d = 768
    x = np.eye(d, dtype=np.float32)
    q = synth(16, d, 3, normalize=False)
    e = _engine(x)
    D, I = e.search(q, 10)
    want = np.argsort(-q, axis=1, kind="stable")[:, :10]
    assert np.array_equal(I, want)
    np.testing.assert_allclose(D, np.take_along_axis(q, want, axis=1), rtol=1e-6)


def test_overflowing_candidate_lists_fall_back_exactly(fo):
    """All-equal corpus: every row ties with the threshold, the candidate lists overflow and
    the queries are re-run on the exact path -- still the right answer (rows 0..k-1)."""
    x = np.tile(synth(1, 256, 5), (20000, 1))
    q = synth(6, 256, 6)
    e = _engine(x)
    D, I = e.search(q, 100, mode="tensor")
    assert e.stats()["fallback_queries"] == 6
    assert np.array_equal(I, np.tile(np.arange(100), (6, 1)))
    Do, Io = fo.search(q, x, 100)
    np.testing.assert_allclose(D, Do, rtol=RTOL)


def test_unnormalised_and_fp16_inputs(fo):
    """Real pipeline data: fp16 arrays (generate_passage_embeddings.py:75-76), not normalised."""
    x = (synth(8000, 768, 11, normalize=False) * 0.3).astype(np.float16)
    q = (synth(40, 768, 12, normalize=False) * 0.3).astype(np.float16)
    e = _engine(x)
    D, I = e.search(q.astype(np.float32), 100)
    Do, Io = fo.search(q.astype(np.float32), x.astype(np.float32), 100)
    fo.compare_topk(D, I, Do, Io, q.astype(np.float32), x.astype(np.float32), rtol=RTOL)
    np.testing.assert_array_equal(e.export_rows(10, 5), x[10:15].astype(np.float32))


def _bf16_round(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).bfloat16().float().numpy()


@pytest.mark.parametrize("mode", ["tensor", "exact"])
@pytest.mark.parametrize("k", [10, 100, 1000])
def test_bf16_storage_is_exact_on_the_stored_values(fo, mode, k):
    """BASELINE config 4: corpus stored in bf16, fp32 rescore.  The oracle sees the
    bf16-rounded rows widened to fp32 -- 'the same inputs'."""
    import torch
    from b2ip import Engine
    x = synth(30000, 768, 51)
    q = synth(48, 768, 52)
    xr = _bf16_round(x)
    e = Engine(768, 0, store="bf16")
    e.add(x[:10000])                                             # fp32 host rows, rounded at ingest
    e.add(torch.from_numpy(x[10000:20000]).cuda())               # fp32 device rows
    e.add(torch.from_numpy(x[20000:]).cuda().bfloat16())         # bf16 device rows
    np.testing.assert_array_equal(e.export_rows(9990, 20), xr[9990:10010])
    np.testing.assert_array_equal(e.export_rows(19990, 20), xr[19990:20010])
    D, I = e.search(q, k, mode=mode)
    Do, Io = fo.search(q, xr, k)
    fo.compare_topk(D, I, Do, Io, q, xr, rtol=RTOL)
    assert e.stats()["fallback_queries"] == 0


def test_bf16_storage_fp16_host_rows_and_rejects_bf16_on_f32_index(fo):
    import torch
    from b2ip import B2ipError, Engine
    x = (synth(5000, 256, 61, normalize=False) * 0.3).astype(np.float16)
    e = Engine(256, 0, store="bf16")
    e.add(x)
    xr = _bf16_round(x.astype(np.float32))
    q = synth(20, 256, 62)
    D, I = e.search(q, 50)
    Do, Io = fo.search(q, xr, 50)
    fo.compare_topk(D, I, Do, Io, q, xr, rtol=RTOL)
    f32 = Engine(256, 0)
    with pytest.raises((B2ipError, KeyError)):
        f32._lib.b2ip_add  # noqa: B018
        import ctypes
        t = torch.zeros((4, 256), dtype=torch.bfloat16, device="cuda")
        from b2ip._lib import B2IP_BF16, MEM_DEVICE, check
        check(f32._lib.b2ip_add(f32._h, 4, ctypes.c_void_p(t.data_ptr()), B2IP_BF16, MEM_DEVICE), f32._h)


@pytest.mark.parametrize("mode", ["tensor", "exact"])
@pytest.mark.parametrize("k", [10, 100, 1000])
def test_f16_storage_is_lossless_for_fp16_shards(fo, mode, k):
    """The reference's default pipeline: float16 shards, widened by astype('float32')
    (src/index.py:27).  An fp16 store keeps exactly those values: the oracle sees x.astype(f32)."""
    import torch
    from b2ip import Engine
    x = (synth(30000, 768, 71, normalize=False) * 0.3).astype(np.float16)
    q = (synth(48, 768, 72, normalize=False) * 0.3).astype(np.float16).astype(np.float32)
    e = Engine(768, 0, store="f16")
    e.add(x[:10000])                                             # fp16 host rows
    e.add(torch.from_numpy(x[10000:20000]).cuda())               # fp16 device rows
    e.add(torch.from_numpy(x[20000:].astype(np.float32)).cuda())  # fp32 rows that are fp16-valued
    x32 = x.astype(np.float32)
    np.testing.assert_array_equal(e.export_rows(9990, 20), x32[9990:10010])
    np.testing.assert_array_equal(e.export_rows(19990, 20), x32[19990:20010])
    D, I = e.search(q, k, mode=mode)
    Do, Io = fo.search(q, x32, k)
    fo.compare_topk(D, I, Do, Io, q, x32, rtol=RTOL)
    st = e.stats()
    assert st["fallback_queries"] == 0
    if mode == "tensor":
        # lossless operands: the error bound is accumulation slack only, so little more than
        # the top-k itself survives to the rescore
        assert st["rescored"] <= 48 * (k + k // 10 + 8)


def test_f16_storage_rounds_fp32_rows_and_saturates(fo):
    """fp32 rows into an fp16 store are rounded to nearest, saturating at +-65504 (no inf is
    ever created); the search is exact on the stored values."""
    from b2ip import Engine
    x = synth(6000, 256, 73, normalize=False)
    x[17, 3] = 1.0e6
    x[18, 5] = -3.0e7
    e = Engine(256, 0, store="f16")
    e.add(x)
    xr = np.clip(x, -65504.0, 65504.0).astype(np.float16).astype(np.float32)
    np.testing.assert_array_equal(e.export_rows(0, 6000), xr)
    q = synth(20, 256, 74)
    D, I = e.search(q, 50)
    Do, Io = fo.search(q, xr, 50)
    fo.compare_topk(D, I, Do, Io, q, xr, rtol=RTOL)


@pytest.mark.parametrize("shadow", ["bf16", "f16"])
def test_shadow_operand_type_of_an_fp32_index(fo, shadow):
    """fp32 master rows with either 16-bit operand type for the coarse pass: same answers; the
    fp16 shadow's tighter bound sends fewer rows to the rescore.  Includes values beyond the
    fp16 range (saturated shadow, bound computed from the stored value)."""
    from b2ip import Engine
    x = synth(40000, 768, 81)
    q = synth(64, 768, 82)
    e = Engine(768, 0, shadow=shadow)
    e.add(x)
    D, I = e.search(q, 100, mode="tensor")
    Do, Io = fo.search(q, x, 100)
    fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)
    st = e.stats()
    assert st["fallback_queries"] == 0
    resc = st["rescored"] / 64
    assert resc < (140 if shadow == "f16" else 400), resc
    if shadow == "f16":
        got = e.debug_coarse_scores(__import__("torch").from_numpy(q).cuda(), 0, 1024).cpu().numpy()
        want = q.astype(np.float16).astype(np.float64) @ x[:1024].astype(np.float16).astype(np.float64).T
        np.testing.assert_allclose(got, want, rtol=0, atol=2e-5)
    # out-of-range values: still exact (the affected queries may take the exact path)
    x2 = x[:5000].copy()
    x2[100] *= 1.0e6
    e2 = Engine(768, 0, shadow=shadow)
    e2.add(x2)
    D, I = e2.search(q[:8], 10)
    Do, Io = fo.search(q[:8], x2, 10)
    fo.compare_topk(D, I, Do, Io, q[:8], x2, rtol=RTOL)


def test_indexer_auto_store_and_migration(fo):
    """Indexer(store='auto'): float16 chunks live in an fp16 store; the first non-fp16 chunk moves
    everything to fp32 master rows.  Results equal the reference restatement either way."""
    from src.index import Indexer
    d, k = 256, 20
    a = (synth(3000, d, 91, normalize=False) * 0.5).astype(np.float16)
    b = (synth(2000, d, 92, normalize=False) * 0.5).astype(np.float16)
    c = synth(1000, d, 93, normalize=False) * 0.5                       # fp32, not fp16-valued
    ours, ref = Indexer(d, 0, 8), fo.OracleIndexer(d, 0, 8)
    for idx in (ours, ref):
        idx.index_data([str(i) for i in range(3000)], a)
        idx.index_data([str(3000 + i) for i in range(2000)], b)
    assert ours.index.store == "f16" and ours.index.ntotal == 5000
    q = (synth(30, d, 94, normalize=False)).astype(np.float16)

    def check():
        got, want = ours.search_knn(q, k), ref.search_knn(q, k)
        fo.compare_topk(np.stack([g[1] for g in got]), np.array([[int(s) for s in g[0]] for g in got]),
                        np.stack([w[1] for w in want]), np.array([[int(s) for s in w[0]] for w in want]),
                        q.astype(np.float32), ref.rows, rtol=RTOL)
    check()
    for idx in (ours, ref):
        idx.index_data([str(5000 + i) for i in range(1000)], c)
    assert ours.index.store == "f32" and ours.index.ntotal == 6000
    np.testing.assert_array_equal(ours.index.export_rows(2990, 20), np.concatenate([a, b])[2990:3010].astype(np.float32))
    check()


def test_incremental_adds_equal_one_add(fo):
    x = synth(7000, 768, 21)
    q = synth(20, 768, 22)
    from b2ip import Engine
    e = Engine(768, 0)
    for a, b in [(0, 1), (1, 300), (300, 4096), (4096, 7000)]:
        e.add(x[a:b])
    assert e.ntotal == 7000
    D, I = e.search(q, 100)
    Do, Io = fo.search(q, x, 100)
    fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)


def test_rows_grow_in_place_and_match_the_copying_fallback(fo):
    """The index grows in place (CUDA virtual memory management: no reserve, no regrowth copy) --
    many small and large appends give the same rows and answers as one add, and as the
    cudaMalloc + copy fallback (B2IP_VMM=0) run in a fresh process."""
    import subprocess
    import sys
    from b2ip import Engine
    x = synth(70_000, 256, 41)
    q = synth(33, 256, 42)
    one = Engine(256, 0)
    one.add(x)
    many = Engine(256, 0)
    cuts = [0, 1, 2, 300, 301, 5000, 5001, 40_000, 70_000]
    for a, b in zip(cuts, cuts[1:]):
        many.add(x[a:b])
    assert many.ntotal == 70_000
    np.testing.assert_array_equal(many.export_rows(0, 70_000), x)
    Da, Ia = one.search(q, 50)
    Db, Ib = many.search(q, 50)
    assert np.array_equal(Ia, Ib) and np.array_equal(Da, Db)
    code = (
        "import sys, numpy as np; sys.path[:0] = %r\n"
        "from helpers import synth; from b2ip import Engine\n"
        "x = synth(70_000, 256, 41); q = synth(33, 256, 42); e = Engine(256, 0)\n"
        "[e.add(x[a:b]) for a, b in zip(%r, %r)]\n"
        "D, I = e.search(q, 50); np.save(sys.argv[1], I); np.save(sys.argv[2], D)\n"
    ) % ([os.path.join(ROOT, "czech-contriever_b200"), os.path.join(ROOT, "tests"), ROOT], cuts[:-1], cuts[1:])
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        fi, fd = os.path.join(td, "I.npy"), os.path.join(td, "D.npy")
        out = subprocess.run([sys.executable, "-c", code, fi, fd], env=dict(os.environ, B2IP_VMM="0"),
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        assert np.array_equal(np.load(fi), Ia) and np.array_equal(np.load(fd), Da)


def test_torch_device_buffers(fo):
    import torch
    x = synth(6000, 768, 31)
    q = synth(70, 768, 32)
    from b2ip import Engine
    e = Engine(768, 0)
    e.add(torch.from_numpy(x).cuda())
    D, I = e.search(torch.from_numpy(q).cuda(), 100)
    Do, Io = fo.search(q, x, 100)
    fo.compare_topk(D.cpu().numpy(), I.cpu().numpy(), Do, Io, q, x, rtol=RTOL)


def test_merge_topk_and_sharded_equals_single(fo):
    """Two row shards on one GPU + merge kernel == one index (the multi-GPU path minus NCCL)."""
    import torch
    from b2ip import Engine, merge_topk
    x = synth(9000, 768, 41)
    q = synth(64, 768, 42)
    k = 100
    whole = _engine(x)
    Dw, Iw = whole.search(q, k)
    parts = []
    for lo, hi in [(0, 4000), (4000, 9000)]:
        e = Engine(768, 0)
        e.add(x[lo:hi])
        e.set_row_offset(lo)
        parts.append(e.search(torch.from_numpy(q).cuda(), k))
    gD = torch.stack([p[0] for p in parts])
    gI = torch.stack([p[1] for p in parts])
    D, I = merge_topk(gD, gI, k)
    assert np.array_equal(I.cpu().numpy(), Iw)
    np.testing.assert_array_equal(D.cpu().numpy(), Dw)


def test_indexer_drop_in(fo, tmp_path):
    """Same calls on the B200 `Indexer` and on the oracle's restatement of the reference one:
    pickle shards -> driver ingest loop -> search_knn -> serialize -> deserialize_from."""
    from src.index import Indexer
    d, k = 768, 100
    shards = []
    start = 0
    for i, n in enumerate([1500, 700, 2300]):
        emb = synth(n, d, 100 + i, normalize=False).astype(np.float16)
        ids = [str(start + j) for j in range(n)]          # str ids, as load_passages yields
        path = tmp_path / f"passages_{i:02d}"
        with open(path, "wb") as f:
            pickle.dump((ids, emb), f)                    # generate_passage_embeddings.py:94-95
        start += n
    files = sorted(str(p) for p in tmp_path.glob("passages_*"))
    for f in files:
        with open(f, "rb") as fin:
            shards.append(pickle.load(fin))
    ours, ref = Indexer(d, 0, 8), fo.OracleIndexer(d, 0, 8)
    ingest_like_reference_driver(ours, shards, 1000)
    ingest_like_reference_driver(ref, shards, 1000)
    assert ours.index_id_to_db_id == ref.index_id_to_db_id
    q = synth(50, d, 777, normalize=False).astype(np.float16)
    got, want = ours.search_knn(q, k), ref.search_knn(q, k)
    assert len(got) == len(want) == 50
    x = ref.rows
    for (gi, gs), (wi, ws) in zip(got, want):
        assert isinstance(gi, list) and isinstance(gi[0], str) and gs.dtype == np.float32
        assert gs.shape == (k,)
    fo.compare_topk(np.stack([g[1] for g in got]), np.array([[int(s) for s in g[0]] for g in got]),
                    np.stack([w[1] for w in want]), np.array([[int(s) for s in w[0]] for w in want]),
                    q.astype(np.float32), x, rtol=RTOL)
    # persistence: our files are readable by the oracle's reader and vice versa
    da, db = tmp_path / "a", tmp_path / "b"
    da.mkdir(); db.mkdir()
    ours.serialize(str(da)); ref.serialize(str(db))
    assert open(da / "index.faiss", "rb").read() == open(db / "index.faiss", "rb").read()
    again = Indexer(d, 0, 8)
    again.deserialize_from(str(db))
    got2 = again.search_knn(q, k)
    for (a, sa), (b, sb) in zip(got, got2):
        assert a == b and np.array_equal(sa, sb)


def test_single_process_multi_engine_equals_one_engine(fo, tmp_path):
    """b2ip.multi.MultiGpuEngine (here: three shards on the one visible GPU) returns exactly what a
    single Engine returns -- ids, scores, ties -- for one-shot and chunked ingest, host and device
    queries, and exports rows by global id."""
    import torch
    from b2ip import Engine, MultiGpuEngine
    x = synth(30_000, 256, 111)
    x[20_000:20_040] = x[5:45]                       # exact ties across shards
    q = synth(90, 256, 112)
    whole = Engine(256, 0)
    whole.add(x)
    for chunks in ([(0, 30_000)], [(0, 7000), (7000, 7001), (7001, 19_000), (19_000, 30_000)]):
        m = MultiGpuEngine(256, [0, 0, 0])
        for a, b in chunks:
            m.add(x[a:b])
        assert m.ntotal == 30_000
        for k in (1, 10, 100):
            Dw, Iw = whole.search(q, k)
            D, I = m.search(q, k)
            assert np.array_equal(I, Iw) and np.array_equal(D, Dw)
            Dt, It = m.search(torch.from_numpy(q).cuda(), k)
            assert np.array_equal(It.cpu().numpy(), Iw) and np.array_equal(Dt.cpu().numpy(), Dw)
        np.testing.assert_array_equal(m.export_rows(6990, 3000), x[6990:9990])
        assert m.stats()["coarse_launches"] >= 3
        m.close()
    # through the drop-in Indexer: device list -> sharded engine, same search_knn output
    from src.index import Indexer
    ids = [f"doc{i}" for i in range(30_000)]
    one, many = Indexer(256, 0, 8, device=0), Indexer(256, 0, 8, device=[0, 0])
    for idx in (one, many):
        idx.index_data(ids[:12_345], x[:12_345])
        idx.index_data(ids[12_345:], x[12_345:])
    ra, rb = one.search_knn(q, 20), many.search_knn(q, 20)
    for (ia, sa), (ib, sb) in zip(ra, rb):
        assert ia == ib and np.array_equal(sa, sb)
    many.serialize(str(tmp_path))
    again = Indexer(256, 0, 8, device=[0, 0])
    again.deserialize_from(str(tmp_path))
    rc = again.search_knn(q, 20)
    for (ia, sa), (ic, sc) in zip(ra, rc):
        assert ia == ic and np.array_equal(sa, sc)


def test_search_knn_takes_device_queries_and_float16(fo):
    """SURVEY 8f N4 through the drop-in: `Indexer.search_knn` given the encoder's output as a CUDA
    tensor (float16 or float32) returns exactly what it returns for the same values as a host
    array, chunked or not; float16 host queries equal their float32 widening (astype is exact)."""
    import torch
    from src.index import Indexer
    x = synth(20_000, 768, 301, normalize=False)
    q16 = synth(300, 768, 302, normalize=False).astype(np.float16)
    ix = Indexer(768, 0, 8, device=0, store="f32")
    ix.index_data([f"d{i}" for i in range(len(x))], x)
    want = ix.search_knn(q16.astype(np.float32), 20)
    ref = fo.OracleIndexer(768, 0, 8)
    ref.index_data([f"d{i}" for i in range(len(x))], x)
    for (gi, gs), (wi, ws) in zip(want[:50], ref.search_knn(q16[:50], 20)):
        assert gi == wi and np.allclose(gs, ws, rtol=RTOL, atol=0)
    for chunk in (16384, 64):
        ix.knn_chunk = chunk
        for queries in (q16, torch.from_numpy(q16).cuda(), torch.from_numpy(q16.astype(np.float32)).cuda(),
                        torch.from_numpy(q16)):
            got = ix.search_knn(queries, 20)
            assert len(got) == len(want)
            for (gi, gs), (wi, ws) in zip(got, want):
                assert gi == wi and np.array_equal(gs, ws) and gs.dtype == np.float32


def test_indexer_rejects_pq():
    from src.index import Indexer
    with pytest.raises(NotImplementedError):
        Indexer(768, 16, 8)


def test_golden_fixture(fo):
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "flatip_small.npz"))
    e = _engine(g["corpus"])
    for k in (1, 10, 100):
        D, I = e.search(g["queries"], k)
        fo.compare_topk(D, I, g[f"D_k{k}"], g[f"I_k{k}"], g["queries"], g["corpus"], rtol=RTOL)


def test_c2_scale_subset(fo):
    """BASELINE config 2 scale (1M x 768, k=100) on the GPU; the oracle checks a fixed random
    subset of queries against the full corpus, every row must be descending and in range."""
    import torch
    n, nq, k, d = 1_000_000, 2048, 100, 768
    gen = torch.Generator(device="cuda").manual_seed(1234)
    x = torch.randn((n, d), generator=gen, device="cuda")
    x /= x.norm(dim=1, keepdim=True)
    gen.manual_seed(4321)
    q = torch.randn((nq, d), generator=gen, device="cuda")
    q /= q.norm(dim=1, keepdim=True)
    from b2ip import Engine
    e = Engine(d, 0)
    e.add(x)
    D, I = e.search(q, k)
    D, I = D.cpu().numpy(), I.cpu().numpy()
    assert (np.diff(D, axis=1) <= 0).all() and I.min() >= 0 and I.max() < n
    assert e.stats()["fallback_queries"] == 0
    sel = np.random.default_rng(0).choice(nq, 64, replace=False)
    xh, qh = x.cpu().numpy(), q[torch.from_numpy(sel).cuda()].cpu().numpy()
    Do, Io = fo.search(qh, xh, k)
    fo.compare_topk(D[sel], I[sel], Do, Io, qh, xh, rtol=RTOL)


@pytest.mark.parametrize("store,shadow", [("f32", "bf16"), ("f32", "f16"), ("f16", None)])
def test_non_finite_values_follow_faiss(fo, store, shadow):
    """NaN / inf in the corpus or in a query (fp16 encoders do overflow): faiss never returns a
    NaN score, returns +inf scores first, and pads a query that scores NaN everywhere.  A row
    with a non-finite element must not poison the error bound of the other rows."""
    from b2ip import Engine
    n, d, k = 20_000, 256, 20
    x = synth(n, d, 131)
    x[11] = np.nan                    # never reported
    x[500, 3] = np.inf                # +inf or -inf score depending on the query's sign there
    x[9000, 7] = -np.inf
    x[15000, 1] = np.inf; x[15000, 2] = -np.inf     # +inf, -inf or NaN (inf - inf) by the query's signs
    q = synth(24, d, 132)
    q[5] = np.nan                     # scores NaN everywhere -> all padding
    if store == "f16":
        x = x.astype(np.float16).astype(np.float32)
    e = Engine(d, 0, store=store, shadow=shadow)
    e.add(x)
    for mode in ("tensor", "exact"):
        D, I = e.search(q, k, mode=mode)
        Do, Io = fo.search(q, x, k)
        assert not np.isnan(D).any()
        assert (I[5] == -1).all() and (D[5] == np.finfo(np.float32).min).all()
        assert np.array_equal(I[5], Io[5])
        assert not np.isin(I, [11]).any()
        assert np.array_equal(np.isposinf(D), np.isposinf(Do))
        rows = [i for i in range(24) if i != 5]
        # rows that score +inf come first, the rest as usual
        for r in rows:                            # (order among equal scores is heap-defined in faiss)
            assert sorted(I[r][np.isposinf(D[r])]) == sorted(Io[r][np.isposinf(Do[r])])
        fin = np.isfinite(Do[rows]).all(axis=1)
        sel = [r for r, f in zip(rows, fin) if f]
        xs = x.copy()
        xs[[11, 500, 9000, 15000]] = 0.0          # tie classification only needs finite rows
        Dm, Im, Dom, Iom = D[rows].copy(), I[rows].copy(), Do[rows].copy(), Io[rows].copy()
        inf_mask = np.isposinf(Dom)
        Dm[inf_mask] = 0; Dom[inf_mask] = 0       # compared above
        fo.compare_topk(Dm, Im, Dom, Iom, q[rows], xs, rtol=RTOL)
    if store == "f32":
        assert e.stats()["mode_used"] == 2
    e2 = Engine(d, 0, store=store, shadow=shadow)
    e2.add(x)
    e2.search(q, k, mode="tensor")
    st = e2.stats()
    # the non-finite rows did not push everything onto the exact path
    assert st["fallback_queries"] <= 1, st


@pytest.mark.parametrize("d,nq", [(2048, 8), (1024, 40), (1024, 20), (64, 64)])
def test_small_batches_across_dimensions(fo, d, nq):
    """Batches <= 64 take the streaming kernel (queries resident in shared memory) when the padded
    batch (32 query rows for <= 32 queries, else 64) fits next to >= 4 corpus stages of 16 KiB:
    d_pad <= 2560 for <= 32 queries, d_pad <= 1280 for 33-64.  All four cases here stream (d = 2048
    with 8 queries: 128 KiB of queries, 6 stages), which the threshold bootstrap's sample shows; the
    single-CTA side of the rule is tested by test_gpu_edges.test_small_batch_kernel_choice."""
    x = synth(30_000, d, 141)
    q = synth(nq, d, 142)
    e = _engine(x)
    D, I = e.search(q, 10)
    assert e.stats()["fallback_queries"] == 0 and e.stats()["slabs"] >= 2
    assert e.stats()["sample_rows"] > 0
    Do, Io = fo.search(q, x, 10)
    fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)
