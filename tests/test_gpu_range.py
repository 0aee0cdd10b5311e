"""Range search on the GPU (`Engine.range_search`, `b2ip_range_search`): every row whose exact score
is strictly above the radius.

Answers are held to an fp64 checker on the stored values with the rescore's rounding bound b of
`test_gpu_edges.check_topk` (tensor path): every returned score within b of its fp64 value and above
the radius, every row certainly above the radius (s64 - b > r) returned, none certainly below
(s64 + b <= r).  Both paths compute scores with the same arithmetic, so the tensor and exact modes
must agree bit for bit, and a row that `search` returns scores the same bits in both."""
import ctypes

import numpy as np
import pytest

from helpers import synth
from test_gpu_edges import U, _gamma_for

gpu = pytest.mark.gpu
F32 = np.float32


@pytest.fixture(scope="module")
def b2ip_mod():
    import __graft_entry__ as g
    g.build()
    import b2ip
    return b2ip


def _engine(b2ip, x, store="f32"):
    e = b2ip.Engine(x.shape[1], 0, store=store)
    e.add(x)
    return e


def _stored(e, x):
    """The values the index holds, as a CUDA fp32 tensor."""
    import torch
    if e.store == "f32":
        return torch.as_tensor(np.asarray(x, F32)).cuda() if not hasattr(x, "is_cuda") else x.float()
    return torch.as_tensor(e.export_rows(0, e.ntotal)).cuda()


def fp64_scores(q, xs, c0, c1):
    """(S, B) for rows [c0, c1): fp64 scores of the stored values and the per-row rounding bound."""
    import torch
    q64 = torch.as_tensor(np.asarray(q, np.float64)).cuda() if not hasattr(q, "is_cuda") else q.double()
    xc = xs[c0:c1].double()
    d = q64.shape[1]
    S = q64 @ xc.T
    A = q64.abs() @ xc.abs().T
    B = (_gamma_for("tensor", d) + d * 2.0 ** -52) * A + U * S.abs()
    return S, B


def check_range(lims, D, I, q, xs, radius):
    """Strict check of a CSR range answer against fp64 scores of the stored values xs (CUDA tensor)."""
    import torch
    lims, D, I = (np.asarray(a) for a in (lims, D, I))
    nq, n = len(lims) - 1, xs.shape[0]
    assert lims.dtype == np.int64 and D.dtype == np.float32 and I.dtype == np.int64
    assert lims[0] == 0 and (np.diff(lims) >= 0).all() and lims[-1] == len(D) == len(I), "lims"
    assert ((I >= 0) & (I < n)).all(), "row out of range"
    qi = np.repeat(np.arange(nq), np.diff(lims))
    same_q = qi[1:] == qi[:-1]
    assert (I[1:][same_q] > I[:-1][same_q]).all(), "rows not unique and ascending"
    assert (D > radius).all(), "score not above the radius"
    chunk = max(256, min((1 << 24) // xs.shape[1], (1 << 25) // max(nq, 1)))
    qi_t = torch.as_tensor(qi).cuda()
    I_t = torch.as_tensor(I).cuda()
    D_t = torch.as_tensor(D).cuda().double()
    for c0 in range(0, n, chunk):
        c1 = min(n, c0 + chunk)
        S, B = fp64_scores(q, xs, c0, c1)
        ret = torch.zeros_like(S, dtype=torch.bool)
        sel = (I_t >= c0) & (I_t < c1)
        ret[qi_t[sel], I_t[sel] - c0] = True
        s, b = S[qi_t[sel], I_t[sel] - c0], B[qi_t[sel], I_t[sel] - c0]
        err = (D_t[sel] - s).abs() - b
        assert not (err > 0).any(), f"score off by {float(err.max())} beyond the bound"
        missed = ~ret & (S - B > radius)
        assert not missed.any(), f"rows certainly above the radius missing: {missed.nonzero()[:5].tolist()}"
        extra = ret & ((S + B <= radius) | S.isnan())
        assert not extra.any(), f"rows certainly below the radius returned: {extra.nonzero()[:5].tolist()}"


def same_answer(a, b):
    return all(np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)) for x, y in zip(a, b))


def kth_radius(q, xs, k):
    """A radius that leaves about k rows per query: the median over queries of the k-th fp64 score."""
    import torch
    S, _ = fp64_scores(q, xs, 0, xs.shape[0])
    kk = min(k, xs.shape[0])
    return float(np.float32(torch.topk(S, kk, dim=1).values[:, -1].median().item()))


# ---------------------------------------------------------------------------- 1 + 2: fp64, tensor == exact
@gpu
@pytest.mark.parametrize("store", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("d", [4, 100, 768, 4096])
def test_against_fp64_and_exact_path(b2ip_mod, store, d):
    import torch
    n = 20000 if d <= 768 else 12000
    x = synth(n, d, seed=100 + d)
    e = _engine(b2ip_mod, x, store)
    xs = _stored(e, x)
    for nq in (1, 7, 129, 300):
        q = synth(nq, d, seed=7 * nq + d)
        S, _ = fp64_scores(q, xs, 0, n)
        radii = [float(S.max().item()) + 1.0, kth_radius(q, xs, 10), kth_radius(q, xs, 1000)]
        for r in radii:
            ans = e.range_search(q, r, mode="tensor")
            st = e.stats()
            assert st["k"] == 0 and st["mode_used"] == 1 and st["coarse_launches"] >= 1
            assert st["bound_violations"] == 0 and st["max_err_over_eps"] < 1.0
            check_range(*ans, q, xs, r)
            ex = e.range_search(q, r, mode="exact")
            assert e.stats()["mode_used"] == 2
            assert same_answer(ans, ex), (store, d, nq, r)
        assert e.range_search(q, radii[0])[0][-1] == 0
        assert e.range_search(q, radii[2])[0][-1] > 100 * nq
    torch.cuda.synchronize()
    e.close()


# ---------------------------------------------------------------------------- 3: consistency with search
@gpu
@pytest.mark.parametrize("store", ["f32", "bf16"])
def test_consistent_with_search(b2ip_mod, store):
    k, nq = 100, 24
    x = synth(60000, 768, seed=3)
    q = synth(nq, 768, seed=4)
    e = _engine(b2ip_mod, x, store)
    D, I = e.search(q, k)
    assert e.stats()["fallback_queries"] == 0
    for i in range(nq):
        s_k = D[i, k - 1]
        r = float(np.nextafter(s_k, F32(-np.inf), dtype=F32))
        lims, RD, RI = e.range_search(q[i:i + 1], r)
        order = np.lexsort((RI, -RD.astype(np.float64)))
        RD, RI = RD[order], RI[order]
        assert len(RD) >= k
        assert np.array_equal(RI[:k], I[i]) and np.array_equal(RD[:k].view(np.uint32), D[i].view(np.uint32)), i
        assert (RD[k:] == s_k).all()
    e.close()


# ---------------------------------------------------------------------------- 4: overflow
@gpu
def test_overflowing_list_takes_the_dense_path(b2ip_mod):
    d = 256
    noise = synth(20000, d, seed=11)
    v = synth(1, d, seed=12)
    x = np.concatenate([noise, np.repeat(v, 6000, axis=0), synth(3000, d, seed=13)])
    q = np.concatenate([v, synth(5, d, seed=14)])
    e = _engine(b2ip_mod, x)
    s_v = float(np.float32(v[0].astype(np.float64) @ v[0].astype(np.float64)))
    r = float(np.nextafter(F32(s_v) - F32(1e-3), F32(-np.inf), dtype=F32))
    ans = e.range_search(q, r)
    st = e.stats()
    assert st["fallback_queries"] > 0 and st["slabs"] >= 2, st
    lims = ans[0]
    assert lims[1] - lims[0] >= 6000
    assert same_answer(ans, e.range_search(q, r, mode="exact"))
    check_range(*ans, q, _stored(e, x), r)
    e.close()


# ---------------------------------------------------------------------------- 5: batches, ids, edges
@gpu
def test_query_batches_and_global_ids(b2ip_mod):
    d = 128
    x = synth(30000, d, seed=21)
    q = synth(300, d, seed=22)
    e = _engine(b2ip_mod, x)
    xs = _stored(e, x)
    r = kth_radius(q, xs, 50)
    one = e.range_search(q, r)
    assert e.stats()["query_batches"] == 1
    e.set_option("cand_budget_mb", 1)                   # 128 queries per batch
    many = e.range_search(q, r)
    assert e.stats()["query_batches"] == 3
    assert same_answer(one, many)
    e.set_option("cand_budget_mb", 6144)

    e.set_row_offset(1000)
    off = e.range_search(q, r)
    assert np.array_equal(off[0], one[0]) and np.array_equal(off[1], one[1]) and np.array_equal(off[2], one[2] + 1000)
    e.set_row_segments([(0, 5, 700), (700, 10000, 30000 - 700)])
    seg = e.range_search(q, r)
    mapped = np.where(one[2] < 700, one[2] + 5, one[2] - 700 + 10000)
    assert np.array_equal(seg[0], one[0]) and np.array_equal(seg[1], one[1]) and np.array_equal(seg[2], mapped)
    # the torch path returns the same answer as CUDA tensors
    import torch
    t = e.range_search(torch.as_tensor(q).cuda(), r)
    assert all(a.is_cuda for a in t)
    assert same_answer([a.cpu().numpy() for a in t], seg)
    e.close()


@gpu
def test_empty_index_no_queries_and_minus_inf(b2ip_mod):
    d = 64
    e = b2ip_mod.Engine(d, 0)
    lims, D, I = e.range_search(synth(5, d, seed=1), 0.0)
    assert lims.tolist() == [0] * 6 and len(D) == 0 and len(I) == 0
    x = synth(1000, d, seed=2)
    e.add(x)
    lims, D, I = e.range_search(np.zeros((0, d), F32), 0.0)
    assert lims.tolist() == [0] and len(D) == 0
    q = synth(3, d, seed=3)
    for mode in ("tensor", "exact"):
        lims, D, I = e.range_search(q, float("-inf"), mode=mode)
        assert lims.tolist() == [0, 1000, 2000, 3000]
        assert (I.reshape(3, 1000) == np.arange(1000)).all()
    e.close()


@gpu
def test_nan_rows_and_inf_queries(b2ip_mod):
    d = 64
    x = synth(5000, d, seed=31)
    x[17, 3] = np.nan
    x[4000, 0] = np.nan
    e = _engine(b2ip_mod, x)
    q = synth(4, d, seed=32)
    lims, D, I = e.range_search(q, float("-inf"))
    assert not np.isin([17, 4000], I).any() and (np.diff(lims) == 4998).all()
    q[2, 5] = np.inf
    ans = e.range_search(q, 0.05)
    assert e.stats()["fallback_queries"] >= 1
    assert same_answer(ans, e.range_search(q, 0.05, mode="exact"))
    e.close()


# ---------------------------------------------------------------------------- 6: arguments, held answer
@gpu
def test_arguments_and_the_held_answer(b2ip_mod):
    from b2ip._lib import B2ipError
    d = 64
    x = synth(4000, d, seed=41)
    q = synth(16, d, seed=42)
    e = _engine(b2ip_mod, x)
    lib, h = e._lib, e._h
    lims = np.zeros(17, np.int64)
    D = np.zeros(100000, F32)
    I = np.zeros(100000, np.int64)
    ptr = lambda a: ctypes.c_void_p(a.ctypes.data)
    assert lib.b2ip_range_fetch(h, ptr(D), ptr(I), 0) == -1              # nothing held yet
    D0, I0 = e.search(q, 50)
    with pytest.raises(B2ipError):
        e.range_search(q, float("nan"))
    assert lib.b2ip_range_search(h, 16, ptr(q), 0, ctypes.c_float(0.1), 7, 0, ptr(lims)) == -1
    assert lib.b2ip_range_search(h, 16, ptr(q), 5, ctypes.c_float(0.1), 0, 0, ptr(lims)) == -1
    assert lib.b2ip_range_search(h, 16, ptr(q), 0, ctypes.c_float(0.1), 0, 3, ptr(lims)) == -1
    assert lib.b2ip_range_search(h, -1, ptr(q), 0, ctypes.c_float(0.1), 0, 0, ptr(lims)) == -1
    ans = e.range_search(q, 0.2)
    assert lib.b2ip_range_fetch(h, ptr(D), ptr(I), 0) == 0
    assert np.array_equal(D[:len(ans[1])], ans[1]) and np.array_equal(I[:len(ans[2])], ans[2])
    D1, I1 = e.search(q, 50)                                               # no shared state disturbed
    assert np.array_equal(D0.view(np.uint32), D1.view(np.uint32)) and np.array_equal(I0, I1)
    e.add(synth(10, d, seed=43))
    assert lib.b2ip_range_fetch(h, ptr(D), ptr(I), 0) == -1              # add released the answer
    assert e.range_search(q, 0.2)[0][-1] >= ans[0][-1]
    e.close()


# ---------------------------------------------------------------------------- 7: shard size
@gpu
def test_shard_size(b2ip_mod):
    import torch
    n, d, nq = 2_600_000, 768, 256
    g = torch.Generator(device="cuda").manual_seed(77)
    x = torch.randn((n, d), generator=g, device="cuda")
    x /= x.norm(dim=1, keepdim=True)
    q = torch.randn((nq, d), generator=g, device="cuda")
    q /= q.norm(dim=1, keepdim=True)
    e = b2ip_mod.Engine(d, 0)
    e.add(x)
    D, _ = e.search(q, 1000)
    r = float(np.float32(D[:, -1].median().item()))
    lims, RD, RI = e.range_search(q, r)
    st = e.stats()
    assert st["bound_violations"] == 0 and st["max_err_over_eps"] < 1.0
    assert 500 * nq < lims[-1].item() < 2000 * nq
    check_range(lims.cpu().numpy(), RD.cpu().numpy(), RI.cpu().numpy(), q, x, r)
    e.close()


# ---------------------------------------------------------------------------- 8: multiple GPUs
@gpu
def test_multi_gpu_equals_one_engine(b2ip_mod):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from b2ip.multi import MultiGpuEngine
    d = 256
    x = synth(40000, d, seed=51)
    q = synth(64, d, seed=52)
    one = _engine(b2ip_mod, x)
    m = MultiGpuEngine(d, [0, 1])
    for c0 in range(0, len(x), 3333):                  # interleaved segments on both shards
        m.add(x[c0:c0 + 3333])
    assert len(m.maps[0].segments) > 1
    r = kth_radius(q, _stored(one, x), 100)
    assert same_answer(m.range_search(q, r), one.range_search(q, r))
    m.close()
    one.close()


# ---------------------------------------------------------------------------- 9: Indexer.search_range
@gpu
def test_indexer_search_range(b2ip_mod):
    import torch
    from b2ip.indexer import Indexer
    d = 768
    x = synth(20000, d, seed=61)
    q = synth(10, d, seed=62)
    idx = Indexer(d, device=0)
    idx.index_data([f"p{i}" for i in range(len(x))], x)
    r = kth_radius(q, _stored(idx.index, x), 30)
    lims, D, I = idx.index.range_search(q, r)
    for qq in (q, q.astype(np.float16), torch.as_tensor(q).cuda()):
        res = idx.search_range(qq, r)
        assert len(res) == len(q)
        if not (isinstance(qq, np.ndarray) and qq.dtype == np.float16):
            for i, (ids, scores) in enumerate(res):
                sl = slice(lims[i], lims[i + 1])
                assert sorted(ids) == sorted(f"p{j}" for j in I[sl])
                assert np.array_equal(np.sort(scores)[::-1], scores)
                assert np.array_equal(np.sort(D[sl])[::-1], scores)
                rows = [int(s[1:]) for s in ids]
                ties = (scores[1:] == scores[:-1])
                assert all(a < b for a, b, t in zip(rows, rows[1:], ties) if t)
        else:
            for ids, scores in res:
                assert (scores > r).all() and np.array_equal(np.sort(scores)[::-1], scores)
