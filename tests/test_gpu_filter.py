"""Filtered search (b2ip_search_filtered, Engine.search(allowed=...)): a search restricted to the
rows an allowed-row mask marks must return exactly what an unfiltered search returns on an Engine
built from those rows alone, with its rows mapped back through np.flatnonzero(mask) -- bit for bit
in D and I whenever neither search sent a query to the exact fallback.  Every answer is also held
to the strict fp64 checker `check_topk` on the allowed rows, every returned id must be allowed, and
every search must report no violation of the coarse error bound."""
import ctypes

import numpy as np
import pytest

from helpers import synth
from test_gpu_edges import OPTION_FLIPS, _sm_count, check_topk

gpu = pytest.mark.gpu
FLT_MAX = float(np.finfo(np.float32).max)


def _engine(x, store="f32"):
    from b2ip import Engine
    e = Engine(x.shape[1], 0, store=store)
    if len(x):
        e.add(x)
    return e


def _stored(e, x):
    return e.export_rows(0, x.shape[0]) if e.store != "f32" and len(x) else x


def _mask(n, kind, k, seed):
    """Allowed-row masks of the patterns the kernels treat differently."""
    rng = np.random.default_rng(seed)
    m = np.zeros(n, bool)
    if isinstance(kind, float):
        m = rng.random(n) < kind
    elif kind == "fewer_than_k":
        m[rng.choice(n, max(1, k // 2), replace=False)] = True
    elif kind == "block":
        m[n // 3:n // 3 + max(3 * k, 500)] = True
    elif kind == "every_32nd":
        m[5::32] = True
    elif kind == "last_tile":                   # only rows of the last, partial 256-row tile
        m[n // 256 * 256:] = True
    else:
        raise ValueError(kind)
    return m


def _oracle(x, store, mask, q, k, mode, opts=()):
    """Unfiltered search of an Engine holding only the allowed rows, rows mapped back."""
    keep = np.flatnonzero(mask)
    o = _engine(x[mask], store)
    for name, value in opts:
        o.set_option(name, value)
    D, I = o.search(q, k, mode=mode)
    st = o.stats()
    o.close()
    if len(keep):
        I = np.where(I >= 0, keep[np.maximum(I, 0)], -1)
    return D, I, st


def _check(e, x, store, q, k, mask, mode="auto", sample=None, opts=(), allowed=None):
    """Filtered search of e against the compacted-index oracle and check_topk; returns (D, I, stats)."""
    D, I = e.search(q, k, mode=mode, allowed=mask if allowed is None else allowed)
    st = e.stats()
    assert st["bound_violations"] == 0, st
    keep = np.flatnonzero(mask)
    assert mask[I[I >= 0]].all(), "a disallowed row was returned"
    Do, Io, so = _oracle(x, store, mask, q, k, mode, opts)
    assert so["bound_violations"] == 0
    if st["fallback_queries"] == 0 and so["fallback_queries"] == 0:
        assert np.array_equal(I, Io), "rows differ from the compacted index's"
        assert np.array_equal(D.view(np.uint32), Do.view(np.uint32)), "scores differ from the compacted index's"
    sel = np.arange(len(q)) if sample is None else sample
    xs = _stored(e, x)[mask]
    Ic = np.where(I >= 0, np.searchsorted(keep, np.maximum(I, 0)), -1)
    if len(keep):
        check_topk(D[sel], Ic[sel], q[sel], xs, k, "exact" if mode == "exact" else "tensor")
    else:
        assert (I == -1).all() and (D == -FLT_MAX).all()
    return D, I, st


# -------------------------------------------------------------------------------- the main matrix
CASES = [
    # store, d, nq, k, mask kind
    ("f32", 768, 1, 10, 0.5), ("f16", 768, 33, 100, 0.01), ("bf16", 768, 64, 10, "block"),
    ("f32", 768, 65, 100, "every_32nd"), ("f16", 768, 300, 10, 0.5), ("bf16", 768, 3000, 10, 0.1),
    ("f32", 4, 1, 1, 0.5), ("f16", 4, 300, 100, "last_tile"), ("bf16", 100, 33, 10, "fewer_than_k"),
    ("f32", 100, 300, 1024, 0.5), ("f16", 100, 1, 2048, 0.5), ("bf16", 100, 65, 2048, "fewer_than_k"),
    ("f32", 4096, 64, 100, 0.01), ("f16", 4096, 129, 10, "block"), ("bf16", 4096, 1, 1024, 0.5),
    ("f32", 768, 300, 100, 0.0), ("bf16", 768, 1, 10, 0.0), ("f32", 768, 64, 10, 1.0),
    ("f16", 768, 300, 1024, "every_32nd"), ("f32", 768, 3000, 100, 0.01),
]


@gpu
@pytest.mark.parametrize("store,d,nq,k,kind", CASES)
def test_filtered_equals_the_compacted_index(store, d, nq, k, kind):
    """Streaming (nq <= 64), single-CTA (65..128), pair (> 128) and adaptive-schedule (> 2048)
    kernels, both modes, all stores, k from 1 to 2048, allowed fractions 1 to 0 and the patterns
    that end a chunk, a tile and a slab differently."""
    n = 8_000 if d == 4096 else 20_000
    x = synth(n, d, 700 + d)
    q = synth(nq, d, 701 + nq)
    mask = _mask(n, kind, k, nq + k)
    e = _engine(x, store)
    sample = None if nq <= 300 else np.random.default_rng(1).choice(nq, 200, replace=False)
    for mode in ("tensor", "exact"):
        D, I, st = _check(e, x, store, q, k, mask, mode, sample)
        if mode == "tensor":
            assert st["mode_used"] == 1 and st["sample_rows"] == 0
        n_ok = int(mask.sum())
        if n_ok < k:
            assert (I[:, n_ok:] == -1).all() and (D[:, n_ok:] == -FLT_MAX).all()
    e.close()


@gpu
def test_junk_bits_past_the_last_row_are_ignored():
    from b2ip._lib import MEM_HOST
    n, d, k = 10_000 + 7, 256, 20
    x = synth(n, d, 711)
    q = synth(40, d, 712)
    mask = np.random.default_rng(3).random(n) < 0.3
    e = _engine(x)
    from b2ip.engine import pack_allowed
    bits = pack_allowed(mask).copy()
    bits[-1] |= np.uint32(0xFFFFFFFF) << np.uint32(n % 32)      # set every bit past row n - 1
    for mode in (1, 2):
        D = np.empty((len(q), k), np.float32)
        I = np.empty((len(q), k), np.int64)
        rc = e._lib.b2ip_search_filtered(e._h, len(q), ctypes.c_void_p(q.ctypes.data), 0, k,
                                         ctypes.c_void_p(bits.ctypes.data), n, ctypes.c_void_p(D.ctypes.data),
                                         ctypes.c_void_p(I.ctypes.data), mode, MEM_HOST)
        assert rc == 0
        assert e.stats()["bound_violations"] == 0
        D0, I0 = e.search(q, k, mode="tensor" if mode == 1 else "exact", allowed=mask)
        assert np.array_equal(I, I0) and np.array_equal(D, D0)
    e.close()


@gpu
@pytest.mark.parametrize("nq", [1, 64, 65, 300])
def test_all_ones_mask_equals_the_unfiltered_search(nq):
    x = synth(30_000, 768, 721)
    q = synth(nq, 768, 722)
    e = _engine(x)
    for mode in ("tensor", "exact"):
        D0, I0 = e.search(q, 100, mode=mode)
        D, I = e.search(q, 100, mode=mode, allowed=np.ones(len(x), bool))
        assert e.stats()["bound_violations"] == 0
        assert np.array_equal(I, I0) and np.array_equal(D.view(np.uint32), D0.view(np.uint32))
    e.close()


@gpu
@pytest.mark.parametrize("nq", [8, 200])
def test_best_rows_disallowed(nq):
    """The 50 best rows of every query are disallowed: none may come back, and the best allowed
    rows must."""
    d, k = 768, 50
    x = synth(40_000, d, 731)
    q = synth(nq, d, 732)
    best = np.argsort(-(q.astype(np.float64) @ x.T.astype(np.float64)), axis=1)[:, :50]
    mask = np.ones(len(x), bool)
    mask[best.ravel()] = False
    e = _engine(x)
    D, I, _ = _check(e, x, "f32", q, k, mask)
    assert not np.isin(I, best).any()
    e.close()


@gpu
def test_overflowing_list_with_a_filter():
    """10,000 copies of one row, every third one disallowed; query 200 is that row, so its list
    overflows and the exact fallback answers it: with the filter, i.e. the first k ALLOWED copies."""
    d, k, nq = 768, 100, 300
    x = synth(50_000, d, 741)
    u = x[7000].copy()
    x[7000:17_000] = u
    q = synth(nq, d, 742)
    q[(q @ u) > 0] *= -1
    q[200] = u
    mask = np.ones(len(x), bool)
    mask[7000:17_000:3] = False
    e = _engine(x)
    D, I, st = _check(e, x, "f32", q, k, mask, sample=np.r_[0:200, 201:300])
    assert st["fallback_queries"] == 1
    copies = np.arange(7000, 17_000)[mask[7000:17_000]]
    assert np.array_equal(I[200], copies[:k])
    Do, Io, _ = _oracle(x, "f32", mask, q, k, "auto")
    rest = np.r_[0:200, 201:300]
    assert np.array_equal(I[rest], Io[rest]) and np.array_equal(D[rest], Do[rest])
    e.close()


@gpu
@pytest.mark.parametrize("nq,d,store,k", [(1, 768, "f32", 10), (33, 1540, "f16", 10), (65, 768, "bf16", 100),
                                          (300, 768, "f32", 100)])
def test_options_do_not_change_the_filtered_answer(nq, d, store, k):
    x = synth(60_000, d, 750 + d)
    q = synth(nq, d, 751 + d)
    mask = np.random.default_rng(nq).random(len(x)) < 0.3
    e = _engine(x, store)
    defaults = {"pair": 1, "stream_kernel": 1, "bootstrap": 1, "dense_first": 1, "fuse_refresh": 1,
                "two_stage": 1, "list_fill_pct": 70, "gx": max(1, _sm_count() // 2), "cand_budget_mb": 6 << 10,
                "graph": 1}
    D0, I0, s0 = _check(e, x, store, q, k, mask)
    assert s0["fallback_queries"] == 0
    for name, value in OPTION_FLIPS:
        e.set_option(name, value)
        D, I = e.search(q, k, allowed=mask)
        st = e.stats()
        e.set_option(name, defaults[name])
        assert st["bound_violations"] == 0
        if name == "cand_budget_mb":
            assert st["query_batches"] == -(-nq // 128)
        if st["fallback_queries"] == 0:
            assert np.array_equal(I, I0) and np.array_equal(D, D0), (name, value)
        else:
            _check(e, x, store, q, k, mask)
    e.close()


@gpu
@pytest.mark.parametrize("segments", [False, True])
def test_ids_are_global_with_row_offset_or_segments(segments):
    """Bits index LOCAL rows; the ids that come back are global."""
    d, n, k = 256, 20_000, 30
    x = synth(n, d, 761)
    q = synth(50, d, 762)
    mask = np.random.default_rng(5).random(n) < 0.2
    e = _engine(x)
    local = {mode: e.search(q, k, mode=mode, allowed=mask) for mode in ("tensor", "exact")}
    if segments:
        e.set_row_segments([(0, 100_000, 5000), (5000, 300_000, 15_000)])
        to_global = lambda r: np.where(r < 5000, r + 100_000, r - 5000 + 300_000)
    else:
        e.set_row_offset(1_000_000)
        to_global = lambda r: r + 1_000_000
    for mode, (D0, I0) in local.items():
        D, I = e.search(q, k, mode=mode, allowed=mask)
        assert e.stats()["bound_violations"] == 0
        assert np.array_equal(I, np.where(I0 >= 0, to_global(I0), -1)) and np.array_equal(D, D0)
    e.close()


@gpu
def test_graph_replays_with_different_masks():
    """A small batch is captured once per shape; replays with other masks of the same length each
    match their own oracle, and the unfiltered graph of the same shape is kept apart.  (The first
    filtered call allocates the bitmap buffer, which retires the graphs captured before it.)"""
    d, n, nq, k = 768, 100_000, 16, 10
    x = synth(n, d, 771)
    q = synth(nq, d, 772)
    e = _engine(x)
    U0, J0 = e.search(q, k)
    rng = np.random.default_rng(6)
    for it, frac in enumerate([0.5, 0.1, 0.9, 0.01]):
        mask = rng.random(n) < frac
        D, I, st = _check(e, x, "f32", q, k, mask)
        assert st["graph_mode"] == (1 if it == 0 else 2), st["graph_mode"]
        U, J = e.search(q, k)
        assert e.stats()["graph_mode"] == (1 if it == 0 else 2)
        assert np.array_equal(J, J0) and np.array_equal(U, U0)
    e.close()


@gpu
@pytest.mark.parametrize("store", ["f32", "bf16"])
def test_nan_rows_allowed_and_disallowed(store):
    d, n, k = 64, 2000, 2000
    x = synth(n, d, 781)
    x[[17, 600, 1500], 3] = np.nan
    q = synth(4, d, 782)
    mask = np.ones(n, bool)
    mask[[600, 9, 10]] = False                    # one NaN row, two ordinary rows
    e = _engine(x, store)
    for mode in ("tensor", "exact"):
        D, I, _ = _check(e, x, store, q, k, mask, mode)
        assert not np.isin([17, 600, 1500, 9, 10], I).any()
        m = n - 5                                  # allowed rows with a score
        assert (I[:, :m] >= 0).all() and (I[:, m:] == -1).all()
    e.close()


@gpu
def test_host_and_device_queries_and_masks():
    import torch
    x = synth(30_000, 384, 791)
    q = synth(70, 384, 792)
    mask = np.random.default_rng(7).random(len(x)) < 0.25
    e = _engine(x)
    D0, I0, _ = _check(e, x, "f32", q, 50, mask)
    qt, mt, mc = torch.from_numpy(q).cuda(), torch.from_numpy(mask).cuda(), torch.from_numpy(mask)
    # a CPU torch mask is moved to where the queries cross the ABI, like a numpy one
    for qq, mm in ((q, mt), (qt, mask), (qt, mt), (qt, mc), (q, mc), (q.astype(np.float16), mask)):
        D, I = e.search(qq, 50, allowed=mm)
        if isinstance(D, torch.Tensor):
            D, I = D.cpu().numpy(), I.cpu().numpy()
        assert e.stats()["bound_violations"] == 0
        if isinstance(qq, np.ndarray) and qq.dtype == np.float16:
            assert mask[I[I >= 0]].all()
            continue
        assert np.array_equal(I, I0) and np.array_equal(D, D0)
    e.close()


@gpu
def test_argument_errors_leave_the_handle_usable():
    from b2ip import B2ipError
    from b2ip._lib import MEM_HOST
    from b2ip.engine import pack_allowed
    d, n = 128, 5000
    x = synth(n, d, 801)
    q = synth(9, d, 802)
    mask = np.random.default_rng(8).random(n) < 0.5
    e = _engine(x)
    D0, I0, _ = _check(e, x, "f32", q, 20, mask)
    bits = pack_allowed(mask)
    D = np.empty((9, 2049), np.float32)
    I = np.empty((9, 2049), np.int64)
    p = lambda a: ctypes.c_void_p(a.ctypes.data) if a is not None else None
    call = lambda nb, b, k=20, mode=0, dt=0, mem=MEM_HOST: e._lib.b2ip_search_filtered(
        e._h, 9, p(q), dt, k, p(b), nb, p(D), p(I), mode, mem)
    assert call(n - 1, bits) == -1 and call(n + 1, bits) == -1          # n_bits != ntotal
    assert call(n, None) == -1                                          # NULL bitmap
    assert call(n, bits, mode=3) == -1
    assert call(n, bits, k=0) == -1 and call(n, bits, k=2049) == -1
    assert call(n, bits, dt=2) == -1 and call(n, bits, mem=2) == -1
    # mem = DEVICE with device queries and outputs but a host bitmap: refused before any copy
    import torch
    from b2ip._lib import MEM_DEVICE
    qt = torch.from_numpy(q).cuda()
    Dt = torch.empty((9, 20), dtype=torch.float32, device="cuda")
    It = torch.empty((9, 20), dtype=torch.int64, device="cuda")
    assert e._lib.b2ip_search_filtered(e._h, 9, ctypes.c_void_p(qt.data_ptr()), 0, 20, p(bits), n,
                                       ctypes.c_void_p(Dt.data_ptr()), ctypes.c_void_p(It.data_ptr()),
                                       0, MEM_DEVICE) == -1
    with pytest.raises(ValueError):
        e.search(q, 20, allowed=mask[:-1])
    with pytest.raises(B2ipError):
        e.search(q, 2049, allowed=mask)
    D1, I1 = e.search(q, 20, allowed=mask)
    assert np.array_equal(I1, I0) and np.array_equal(D1, D0)
    U0, J0 = e.search(q, 20)
    check_topk(U0, J0, q, x, 20, "tensor")
    e.close()
    empty = _engine(np.zeros((0, d), np.float32))
    D, I = empty.search(q, 5, allowed=np.zeros(0, bool))
    assert (I == -1).all() and (D == -FLT_MAX).all()
    empty.close()


@gpu
@pytest.mark.parametrize("frac", [0.1, 0.001])
def test_shard_size(frac):
    """One 2.6M x 768 shard; a sample of queries checked against fp64 on the allowed rows."""
    import torch
    from b2ip import Engine
    n, d, nq, k = 2_600_000, 768, 256, 100
    g = torch.Generator(device="cuda").manual_seed(81)
    x = torch.randn((n, d), generator=g, device="cuda")
    x /= x.norm(dim=1, keepdim=True)
    q = torch.randn((nq, d), generator=g, device="cuda")
    q /= q.norm(dim=1, keepdim=True)
    mask = torch.rand(n, generator=g, device="cuda") < frac
    e = Engine(d, 0)
    e.add(x)
    D, I = e.search(q, k, allowed=mask)
    st = e.stats()
    assert st["bound_violations"] == 0 and st["max_err_over_eps"] < 1.0
    D, I, m = D.cpu().numpy(), I.cpu().numpy(), mask.cpu().numpy()
    assert m[I[I >= 0]].all()
    keep = np.flatnonzero(m)
    xa = x[mask].cpu().numpy()
    sel = np.arange(0, nq, 8)
    Ic = np.where(I >= 0, np.searchsorted(keep, np.maximum(I, 0)), -1)
    check_topk(D[sel], Ic[sel], q.cpu().numpy()[sel], xa, k, "tensor")
    e.close()


@gpu
@pytest.mark.parametrize("devices", [[0, 0], [0, 1]])
def test_multi_gpu_engine_equals_one_engine(devices):
    import torch
    if len(set(devices)) > torch.cuda.device_count():
        pytest.skip("needs 2 GPUs")
    from b2ip.multi import MultiGpuEngine
    d, k = 256, 100
    x = synth(40_000, d, 811)
    q = synth(64, d, 812)
    mask = np.random.default_rng(9).random(len(x)) < 0.3
    one = _engine(x)
    D0, I0 = one.search(q, k, allowed=mask)
    m = MultiGpuEngine(d, devices)
    for c0 in range(0, len(x), 3333):                  # interleaved segments on both shards
        m.add(x[c0:c0 + 3333])
    assert len(m.maps[0].segments) > 1
    D, I = m.search(q, k, allowed=mask)
    assert np.array_equal(I, I0) and np.array_equal(D, D0)
    assert all(s["bound_violations"] == 0 for s in m.stats()["per_device"])
    Dt, It = m.search(torch.from_numpy(q).cuda(), k, allowed=torch.from_numpy(mask).cuda())
    assert np.array_equal(It.cpu().numpy(), I0) and np.array_equal(Dt.cpu().numpy(), D0)
    m.close()
    one.close()


@gpu
def test_indexer_search_knn_allowed_ids():
    from b2ip.indexer import Indexer
    d = 768
    x = synth(20_000, d, 821)
    q = synth(12, d, 822)
    ids = [f"p{i}" for i in range(len(x))]
    rng = np.random.default_rng(10)
    allowed = sorted(rng.choice(len(x), 3000, replace=False).tolist())
    idx = Indexer(d, device=0)
    idx.index_data(ids, x)
    sub = Indexer(d, device=0)
    sub.index_data([ids[i] for i in allowed], x[allowed])
    got = idx.search_knn(q, 40, allowed_ids=[ids[i] for i in allowed] + ["unknown"])
    want = sub.search_knn(q, 40)
    assert idx.index.stats()["bound_violations"] == 0
    for (gi, gs), (wi, ws) in zip(got, want):
        assert gi == wi and np.array_equal(gs, ws)
    # fewer allowed passages than top_docs: only the real results come back
    few = idx.search_knn(q, 40, allowed_ids=["p5", "p7", "p5"])
    assert all(sorted(i) == ["p5", "p7"] and len(s) == 2 for i, s in few)
