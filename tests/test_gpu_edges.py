"""Edges of the search contract that the parity suite does not reach: k above 1024 (lists of 4k
keys refreshed out of L2, more survivors than the finalize sort buffer, merges of world*k keys),
dimensions that are not multiples of 64 and up to B2IP_MAX_D, the small-batch kernel choice, every
option that must not change the answer, and an overflowing query in a later query batch.

Every result is held to `check_topk`, a strict fp64 checker: each returned score must lie within
an a-priori rounding bound of the fp64 dot product of its own row, and no row left out may score
certainly above the k-th returned score.  Its CPU tests (no `gpu` marker) show which wrong answers
it rejects."""
import ctypes

import numpy as np
import pytest

from helpers import synth

gpu = pytest.mark.gpu
RTOL = 1e-5
FLT_MAX = float(np.finfo(np.float32).max)
U = 2.0 ** -24                       # unit roundoff of fp32


# ------------------------------------------------------------------------------ strict checker
def _gamma(n):
    return n * U / (1.0 - n * U)


def _gamma_for(path, d):
    """Rounding-error factor of one rescored score.  tensor: four products summed in fp32 (one
    multiply + three FMAs) per partial, partials accumulated in fp64.  exact: a chain of
    4*ceil(d/128) fp32 FMAs per lane, then a 5-level fp32 warp sum."""
    if path == "tensor":
        return _gamma(4)
    if path == "exact":
        return _gamma(4 * (-(-d // 128)) + 5)
    raise ValueError(path)


def _row_fingerprints(xs, rows_per_chunk):
    """A 64-bit hash of the bytes of every row (bit-identical rows hash alike)."""
    n, d = xs.shape
    w = np.random.default_rng(12345).integers(1, 2 ** 63, size=d, dtype=np.uint64) | np.uint64(1)
    fp = np.empty(n, dtype=np.uint64)
    for c0 in range(0, n, rows_per_chunk):
        bits = np.ascontiguousarray(xs[c0:c0 + rows_per_chunk], dtype=np.float32).view(np.uint32)
        with np.errstate(over="ignore"):
            fp[c0:c0 + rows_per_chunk] = (bits.astype(np.uint64) * w).sum(axis=1, dtype=np.uint64)
    return fp


def check_topk(D, I, q, xs, k, path):
    """Strict check of a top-k answer.  D [nq,k] float32, I [nq,k] int64; q [nq,d] the queries;
    xs [n,d] the values the index stores (export_rows of a 16-bit store, the fp32 rows otherwise);
    path "tensor" or "exact" selects the rounding bound b(q, row) = gamma * sum|q_i x_i| +
    2^-24 |s64| (+ d * 2^-52 * sum|q_i x_i| for the fp64 sums here and in the kernel).

    Per query: the number of returned rows is min(k, rows with a non-NaN score) and the tail is
    (-FLT_MAX, -1); ids are in range and unique; |D - s64(row)| <= b for every returned pair;
    (-D, I) strictly increases; every row not returned has s64 - b <= the last returned score;
    a returned row's bit-identical lower copies are returned too, with the same score."""
    D = np.asarray(D)
    I = np.asarray(I)
    assert D.dtype == np.float32 and I.dtype == np.int64, (D.dtype, I.dtype)
    q64 = np.asarray(q, dtype=np.float64)
    nq, d = q64.shape
    n = xs.shape[0]
    assert D.shape == (nq, k) and I.shape == (nq, k), (D.shape, I.shape, nq, k)
    gamma = _gamma_for(path, d)
    slack = d * 2.0 ** -52

    valid = I >= 0
    assert ((I == -1) | (valid & (I < n))).all(), "id out of range"
    m = valid.sum(axis=1)
    assert np.array_equal(valid, np.arange(k)[None, :] < m[:, None]), \
        f"padding inside the returned rows (queries {np.nonzero((valid != (np.arange(k)[None, :] < m[:, None])).any(1))[0][:5]})"
    assert (D[~valid] == -FLT_MAX).all(), "padding score is not -FLT_MAX"
    srt = np.sort(np.where(valid, I, -1 - np.arange(k)[None, :]), axis=1)
    dup = (np.diff(srt, axis=1) == 0).any(axis=1)
    assert not dup.any(), f"duplicated id in query {np.nonzero(dup)[0][0]}"
    both = valid[:, 1:]
    desc = (D[:, :-1] > D[:, 1:]) | ((D[:, :-1] == D[:, 1:]) & (I[:, :-1] < I[:, 1:]))
    bad = both & ~desc
    if bad.any():
        qi, j = np.argwhere(bad)[0]
        raise AssertionError(f"order: q={qi} rank {j}: ({D[qi, j]!r}, {I[qi, j]}) before ({D[qi, j + 1]!r}, {I[qi, j + 1]})")

    qa = np.abs(q64)
    rows_per_chunk = max(256, min((1 << 24) // max(d, 1), (1 << 23) // max(nq, 1)))
    s_ret = np.full((nq, k), np.nan)
    b_ret = np.full((nq, k), np.nan)
    non_nan = np.zeros(nq, dtype=np.int64)
    missed = np.full(nq, -np.inf)             # max over rows not returned of s64 - b
    missed_row = np.full(nq, -1)
    for c0 in range(0, n, rows_per_chunk):
        c1 = min(n, c0 + rows_per_chunk)
        xc = np.asarray(xs[c0:c1], dtype=np.float64)
        S = q64 @ xc.T
        A = qa @ np.abs(xc).T
        B = (gamma + slack) * A + U * np.abs(S)
        non_nan += (~np.isnan(S)).sum(axis=1)
        qi, j = np.nonzero(valid & (I >= c0) & (I < c1))
        r = I[qi, j] - c0
        s_ret[qi, j] = S[qi, r]
        b_ret[qi, j] = B[qi, r]
        low = S - B
        low[qi, r] = -np.inf
        low[np.isnan(low)] = -np.inf
        arg = low.argmax(axis=1)
        best = low[np.arange(nq), arg]
        upd = best > missed
        missed[upd] = best[upd]
        missed_row[upd] = arg[upd] + c0
    want_m = np.minimum(k, non_nan)
    if not np.array_equal(m, want_m):
        qi = np.nonzero(m != want_m)[0][0]
        raise AssertionError(f"q={qi}: {m[qi]} rows returned, {want_m[qi]} expected")
    err = np.where(valid, np.abs(D.astype(np.float64) - s_ret), 0.0)
    over = valid & ~(err <= b_ret)
    if over.any():
        qi, j = np.argwhere(over)[0]
        raise AssertionError(f"score: q={qi} rank {j} row {I[qi, j]}: {D[qi, j]!r} vs fp64 {s_ret[qi, j]!r}, "
                             f"bound {b_ret[qi, j]:.3g}")
    kth = np.where(m > 0, D[np.arange(nq), np.maximum(m - 1, 0)].astype(np.float64), np.inf)
    lost = missed > kth
    if lost.any():
        qi = np.nonzero(lost)[0][0]
        raise AssertionError(f"missed: q={qi} row {missed_row[qi]} scores certainly above the k-th returned "
                             f"score {kth[qi]!r} (fp64 score minus bound {missed[qi]!r})")

    # ties: a returned row with bit-identical lower copies must come with all of them
    fp = _row_fingerprints(xs, rows_per_chunk)
    order = np.argsort(fp, kind="stable")               # within a run of equal hashes: ascending rows
    sfp = fp[order]
    run_start = np.r_[0, np.nonzero(sfp[1:] != sfp[:-1])[0] + 1]
    start_of = np.empty(n, dtype=np.int64)
    rank = np.zeros(n, dtype=np.int64)
    if n:
        starts = np.zeros(n, dtype=np.int64)
        starts[run_start] = run_start
        starts = np.maximum.accumulate(starts)
        start_of[order] = starts
        rank = np.empty(n, dtype=np.int64)
        rank[order] = np.arange(n) - starts
    for qi in range(nq):
        ids = I[qi, :m[qi]]
        ranked = ids[rank[ids] > 0]
        if ranked.size == 0:
            continue
        pos = {int(r): j for j, r in enumerate(ids)}
        xsr = np.asarray(xs)
        for r in ranked.tolist():
            for lo in order[start_of[r]:start_of[r] + rank[r]].tolist():
                if lo >= r or not np.array_equal(xsr[lo].view(np.uint32), xsr[r].view(np.uint32)):
                    continue
                assert lo in pos, f"tie: q={qi} returns row {r} but not its identical lower copy {lo}"
                assert D[qi, pos[lo]] == D[qi, pos[r]], \
                    f"tie: q={qi} identical rows {lo} and {r} scored {D[qi, pos[lo]]!r} and {D[qi, pos[r]]!r}"
    return {"queries": nq, "max_err_over_bound": float(np.nanmax(np.where(valid, err / np.maximum(b_ret, 1e-300), 0.0),
                                                              initial=0.0))}


# --------------------------------------------------------------------- CPU tests of the checker
def _fp64_answer(q, x, k):
    """Top-k of the fp64 scores rounded once to fp32, ordered by (score desc, row asc)."""
    s32 = (np.asarray(q, np.float64) @ np.asarray(x, np.float64).T).astype(np.float32)
    nq, n = s32.shape
    kk = min(k, n)
    D = np.full((nq, k), -FLT_MAX, dtype=np.float32)
    I = np.full((nq, k), -1, dtype=np.int64)
    for i in range(nq):
        o = np.lexsort((np.arange(n), -s32[i].astype(np.float64)))[:kk]
        D[i, :kk] = s32[i, o]
        I[i, :kk] = o
    return D, I


@pytest.fixture(scope="module")
def toy():
    x = synth(3000, 64, 5)
    x[2000:2005] = x[100]                          # bit-identical copies of row 100
    q = synth(6, 64, 6)
    q[0] = x[100] + 0.01 * synth(1, 64, 7)[0]      # query 0 returns row 100 and its copies first
    k = 20
    D, I = _fp64_answer(q, x, k)
    assert list(I[0, :6]) == [100, 2000, 2001, 2002, 2003, 2004]
    return q, x, k, D, I


@pytest.mark.parametrize("path", ["tensor", "exact"])
def test_checker_accepts_the_fp64_answer(toy, path):
    q, x, k, D, I = toy
    check_topk(D, I, q, x, k, path)
    # fewer rows than k: padded tail
    Dp, Ip = _fp64_answer(q, x[:7], k)
    check_topk(Dp, Ip, q, x[:7], k, path)


def _rejects(D, I, q, x, k, match):
    with pytest.raises(AssertionError, match=match):
        check_topk(D, I, q, x, k, "tensor")


def test_checker_rejects_a_duplicated_id(toy):
    q, x, k, D, I = toy
    D2, I2 = D.copy(), I.copy()
    I2[1, 6] = I2[1, 5]
    D2[1, 6] = D2[1, 5]
    _rejects(D2, I2, q, x, k, "duplicated")


def test_checker_rejects_swapped_ids(toy):
    q, x, k, D, I = toy
    D2, I2 = D.copy(), I.copy()
    assert D2[2, 3] != D2[2, 9]
    I2[2, [3, 9]] = I2[2, [9, 3]]
    _rejects(D2, I2, q, x, k, "score")


def test_checker_rejects_a_replaced_id(toy):
    q, x, k, D, I = toy
    D2, I2 = D.copy(), I.copy()
    s = q[3].astype(np.float64) @ x.astype(np.float64).T
    I2[3, 4] = int(np.argsort(s)[1500])            # a row from the middle of the ranking
    _rejects(D2, I2, q, x, k, "score")


def test_checker_rejects_a_score_off_by_three_bounds(toy):
    q, x, k, D, I = toy
    r = int(I[4, 0])
    a = np.abs(q[4].astype(np.float64)) @ np.abs(x[r].astype(np.float64))
    s = q[4].astype(np.float64) @ x[r].astype(np.float64)
    b = (_gamma(4) + 64 * 2.0 ** -52) * a + U * abs(s)
    D2 = D.copy()
    D2[4, 0] = np.float32(s + 3 * b)
    assert D2[4, 0] > D[4, 0]
    _rejects(D2, I, q, x, k, "score")
    # ... while a score moved by half a bound passes
    D3 = D.copy()
    D3[4, 0] = np.float32(s + 0.5 * b)
    check_topk(D3, I, q, x, k, "tensor")


def test_checker_rejects_identical_rows_out_of_order(toy):
    q, x, k, D, I = toy
    I2 = I.copy()
    I2[0, [1, 2]] = I2[0, [2, 1]]                  # rows 2000 and 2001, same score, wrong order
    _rejects(D, I2, q, x, k, "order")
    # a higher copy returned in place of a lower one (the set is wrong, the order is not)
    x2 = x.copy()
    x2[2900] = x[100]
    D3, I3 = _fp64_answer(q, x2, 5)                # rows 100, 2000 .. 2003
    assert list(I3[0]) == [100, 2000, 2001, 2002, 2003]
    I4 = I3.copy()
    I4[0, 4] = 2900
    _rejects(D3, I4, q, x2, 5, "tie")


def test_checker_rejects_padding_inside_a_row(toy):
    q, x, k, D, I = toy
    D2, I2 = D.copy(), I.copy()
    I2[5, 7] = -1
    D2[5, 7] = -FLT_MAX
    _rejects(D2, I2, q, x, k, "padding")


def test_checker_rejects_a_missing_row(toy):
    q, x, k, D, I = toy
    # the k-th row replaced by the (k+5)-th, with its correct score: the order and every pair are
    # right, but the row that was dropped scores certainly above the new last score
    Dk, Ik = _fp64_answer(q, x, k + 5)
    D2, I2 = D.copy(), I.copy()
    D2[1, k - 1], I2[1, k - 1] = Dk[1, k + 4], Ik[1, k + 4]
    _rejects(D2, I2, q, x, k, "missed")
    # too few rows returned
    D3, I3 = D.copy(), I.copy()
    D3[1, k - 1], I3[1, k - 1] = -FLT_MAX, -1
    _rejects(D3, I3, q, x, k, "rows returned")


# ------------------------------------------------------------------------------ GPU helpers
@pytest.fixture(scope="module")
def fo():
    from oracle import flatip_oracle
    return flatip_oracle


def _engine(x, store="f32", shadow=None):
    from b2ip import Engine
    e = Engine(x.shape[1], 0, store=store, shadow=shadow)
    e.add(x)
    return e


def _stored(e, x):
    return e.export_rows(0, x.shape[0]) if e.store != "f32" else x


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _check_tensor_stats(st):
    assert st["mode_used"] == 1 and st["bound_violations"] == 0 and st["max_err_over_eps"] < 1.0, st


# --------------------------------------------------------------------------- A. k above 1024
@gpu
@pytest.mark.parametrize("k,store,nq", [
    (1025, "f32", 1), (1025, "f16", 129), (1025, "bf16", 300), (1025, "bf16", 48),
    (1536, "f16", 1), (1536, "f32", 48), (1536, "bf16", 129), (1536, "f32", 300),
    (2048, "bf16", 1), (2048, "f16", 48), (2048, "f32", 129), (2048, "f16", 300),
])
def test_large_k(fo, k, store, nq):
    """Lists of 4k keys (k > 1024) refreshed out of L2 with in-place compaction, on the streaming
    (nq <= 64), pair (nq > 128) and single-CTA kernels, and the exact path's radix select at k."""
    x = synth(30_000, 256, 201)
    q = synth(nq, 256, 202)
    e = _engine(x, store)
    xs = _stored(e, x)
    Do, Io = fo.search(q, xs, k)
    for mode in ("tensor", "exact"):
        D, I = e.search(q, k, mode=mode)
        st = e.stats()
        assert st["fallback_queries"] == 0 and st["k"] == k
        if mode == "tensor":
            _check_tensor_stats(st)
            assert st["slabs"] >= 2
        check_topk(D, I, q, xs, k, mode)
        fo.compare_topk(D, I, Do, Io, q, xs, rtol=RTOL)


@gpu
def test_large_k_more_survivors_than_the_sort_buffer(fo):
    """k = 2048: a handful of rows scaled x2.5 raise max||x||, which widens every query's coarse
    error bound, so more than SORT_CAP = 4096 rows per query survive the last refresh.  The
    finalize kernel then skips the two-stage rescore, rescores them all and radix-selects the k
    best out of global memory before the sort.  8192 rows = one dense slab = the list capacity
    4k: the lists cannot overflow."""
    d, n, nq, k = 4096, 8192, 48, 2048
    x = synth(n, d, 211)
    x[[7, 900, 3000, 5555, 8000]] *= 2.5
    q = synth(nq, d, 212)
    e = _engine(x)
    D, I = e.search(q, k, mode="tensor")
    st = e.stats()
    assert st["fallback_queries"] == 0 and st["slabs"] == 1
    assert st["rescored"] > 4096 * nq, st["rescored"] / nq
    _check_tensor_stats(st)
    check_topk(D, I, q, x, k, "tensor")
    Do, Io = fo.search(q, x, k)
    fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)


@gpu
@pytest.mark.parametrize("store", ["f32", "f16", "bf16"])
def test_large_k_fewer_rows_than_k(fo, store):
    x = synth(1500, 256, 221)
    q = synth(5, 256, 222)
    e = _engine(x, store)
    xs = _stored(e, x)
    for mode in ("tensor", "exact"):
        D, I = e.search(q, 2048, mode=mode)
        assert (I[:, 1500:] == -1).all() and (D[:, 1500:] == -FLT_MAX).all()
        assert e.stats()["fallback_queries"] == 0
        check_topk(D, I, q, xs, 2048, mode)


@gpu
def test_large_k_graph_replay_is_bit_identical():
    x = synth(30_000, 256, 231)
    q = synth(64, 256, 232)
    e = _engine(x)
    e.set_option("graph", 0)
    D0, I0 = e.search(q, 2048)
    s0 = e.stats()
    assert s0["graph_mode"] == 0 and s0["fallback_queries"] == 0
    check_topk(D0, I0, q, x, 2048, "tensor")
    e.set_option("graph", 1)
    for it in range(3):
        D, I = e.search(q, 2048)
        st = e.stats()
        assert st["graph_mode"] == (1 if it == 0 else 2)
        assert np.array_equal(I, I0) and np.array_equal(D, D0)
        assert st["rescored"] == s0["rescored"] and st["candidates"] == s0["candidates"]


@gpu
def test_k_above_the_maximum_is_rejected_and_the_handle_survives(fo):
    from b2ip import MAX_K, B2ipError
    assert MAX_K == 2048
    x = synth(5000, 256, 241)
    q = synth(9, 256, 242)
    e = _engine(x)
    for mode in ("tensor", "exact"):
        with pytest.raises(B2ipError):
            e.search(q, 2049, mode=mode)
    D, I = e.search(q, 2048)
    check_topk(D, I, q, x, 2048, "tensor")
    D, I = e.search(q, 10)
    check_topk(D, I, q, x, 10, "tensor")
    Do, Io = fo.search(q, x, 10)
    fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)


# ------------------------------------------------------------------------ B. merges at k = 2048
@gpu
def test_merge_at_k_2048_equals_one_engine():
    """Two row shards merged by merge_topk (2k keys per query), and MultiGpuEngine over two shards
    of one GPU, must return exactly one engine's answer; identical rows sit in both shards."""
    import torch
    from b2ip import Engine, MultiGpuEngine, merge_topk
    d, k, n, cut = 256, 2048, 20_000, 9000
    x = synth(n, d, 251)
    x[15_000:15_300] = x[100:400]                  # copies across the shard boundary
    q = synth(64, d, 252)
    q[0] = x[150]
    q[1] = x[120] + x[15_210]
    whole = _engine(x)
    Dw, Iw = whole.search(q, k)
    check_topk(Dw, Iw, q, x, k, "tensor")
    assert 150 in Iw[0] and 15_050 in Iw[0]
    qd = torch.from_numpy(q).cuda()
    parts = []
    for lo, hi in [(0, cut), (cut, n)]:
        e = Engine(d, 0)
        e.add(x[lo:hi])
        e.set_row_offset(lo)
        parts.append(e.search(qd, k))
    D, I = merge_topk(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]), k)
    assert np.array_equal(I.cpu().numpy(), Iw) and np.array_equal(D.cpu().numpy(), Dw)
    m = MultiGpuEngine(d, [0, 0])
    m.add(x)
    D, I = m.search(q, k)
    assert np.array_equal(I, Iw) and np.array_equal(D, Dw)
    Dt, It = m.search(qd, k)
    assert np.array_equal(It.cpu().numpy(), Iw) and np.array_equal(Dt.cpu().numpy(), Dw)
    m.close()


# ------------------------------------------------------------------------------ C. dimensions
DIMS = [4, 12, 100, 772, 1000, 1028, 1540, 2052, 4092, 4096]
NQ_FOR_D = {4: 20, 12: 150, 100: 33, 772: 70, 1000: 150, 1028: 20, 1540: 40, 2052: 8, 4092: 130, 4096: 64}


@gpu
@pytest.mark.parametrize("store", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("d", DIMS)
def test_dimensions_not_multiple_of_64(fo, d, store):
    """d_pad != d: zero padding of queries and rows, TMA boxes over padded rows, the 16-bit
    rescore's guards, d > 1024 (query slice from shared memory), the exact path at up to B2IP_MAX_D."""
    nq, k = NQ_FOR_D[d], 50
    x = synth(6000, d, 300 + d)
    q = synth(nq, d, 301 + d)
    e = _engine(x, store)
    xs = _stored(e, x)
    Do, Io = fo.search(q, xs, k)
    for mode in ("tensor", "exact"):
        D, I = e.search(q, k, mode=mode)
        st = e.stats()
        assert st["fallback_queries"] == 0
        if mode == "tensor":
            _check_tensor_stats(st)
            assert st["slabs"] >= 2
        check_topk(D, I, q, xs, k, mode)
        fo.compare_topk(D, I, Do, Io, q, xs, rtol=RTOL)


@gpu
@pytest.mark.parametrize("store", ["f32", "f16", "bf16"])
def test_positive_data_at_the_largest_dimension(fo, store):
    """Long same-sign sums with the largest accumulation slack d_pad * 2^-23 of the coarse bound."""
    d, k = 4096, 50
    x = np.abs(synth(6000, d, 311))
    q = np.abs(synth(64, d, 312))
    e = _engine(x, store)
    xs = _stored(e, x)
    for nq in (64, 200):
        qq = np.abs(synth(nq, d, 313)) if nq != 64 else q
        D, I = e.search(qq, k, mode="tensor")
        st = e.stats()
        assert st["fallback_queries"] == 0
        _check_tensor_stats(st)
        check_topk(D, I, qq, xs, k, "tensor")
    D, I = e.search(q, k, mode="exact")
    check_topk(D, I, q, xs, k, "exact")


@gpu
@pytest.mark.parametrize("shadow", ["bf16", "f16"])
@pytest.mark.parametrize("d", DIMS)
def test_coarse_scores_padding_adds_nothing(d, shadow):
    """The tcgen05 mainloop alone at d_pad != d: raw scores equal an fp64 product of the rounded
    operands, so the zero padding of queries and rows contributes nothing."""
    import torch
    x = synth(1000, d, 320 + d)
    q = synth(37, d, 321 + d)
    e = _engine(x, shadow=shadow)
    qt = torch.from_numpy(q).cuda()
    got = e.debug_coarse_scores(qt, 0, 1000).cpu().numpy()
    if shadow == "f16":
        want = q.astype(np.float16).astype(np.float64) @ x.astype(np.float16).astype(np.float64).T
    else:
        want = qt.bfloat16().double().cpu().numpy() @ torch.from_numpy(x).bfloat16().double().numpy().T
    np.testing.assert_allclose(got, want, rtol=0, atol=2e-5)


@gpu
@pytest.mark.parametrize("d", [2, 6, 4100, 0])
def test_unsupported_dimensions_are_rejected(d):
    from b2ip import B2ipError, Engine
    for store in ("f32", "f16", "bf16"):
        with pytest.raises(B2ipError):
            Engine(d, 0, store=store)


# ------------------------------------------------------------ D. kernel choice of small batches
def _streams(d, nq):
    """The rule of tensor_search: a batch of <= 64 queries runs the streaming kernel when its
    padded queries (32 or 64 rows of d_pad 16-bit values) leave room for >= 4 corpus stages of
    16 KiB in 227 KiB of shared memory (1344 B reserved); the single-CTA kernel otherwise."""
    d_pad = -(-d // 64) * 64
    q_bytes = d_pad * 2 * (32 if nq <= 32 else 64)
    return nq <= 64 and (227 * 1024 - 1344 - q_bytes) // (128 * 128) >= 4


@gpu
@pytest.mark.parametrize("d,nq,stream", [(1536, 40, False), (4096, 8, False), (1536, 20, True), (2048, 8, True),
                                         (1280, 64, True), (1344, 33, False), (2560, 32, True), (2624, 1, False)])
def test_small_batch_kernel_choice(fo, d, nq, stream):
    """Which kernel a batch of <= 64 queries runs is observable: with the threshold bootstrap on and
    a corpus its planner accepts, the bootstrap runs (sample_rows > 0, the planned sample) exactly
    when the streaming kernel does."""
    assert _streams(d, nq) == stream
    n, k = 30_000, 10
    import b2ip
    lib = b2ip.load()
    grid, tiles = ctypes.c_int32(-1), ctypes.c_int64(-1)
    assert lib.b2ip_debug_plan_bootstrap(n, k, 4096, _sm_count(), -(-d // 64) * 64, 64,
                                         ctypes.byref(grid), ctypes.byref(tiles)) == 0
    assert grid.value > 0, "the planner must accept this corpus"
    x = synth(n, d, 400 + d)
    q = synth(nq, d, 401 + d)
    e = _engine(x)
    D, I = e.search(q, k)
    st = e.stats()
    assert st["fallback_queries"] == 0
    _check_tensor_stats(st)
    assert st["sample_rows"] == (tiles.value * 128 if stream else 0), (st["sample_rows"], tiles.value)
    check_topk(D, I, q, x, k, "tensor")
    Do, Io = fo.search(q, x, k)
    fo.compare_topk(D, I, Do, Io, q, x, rtol=RTOL)


# -------------------------------------------------------------------------- E. option matrix
OPTION_FLIPS = [("pair", 0), ("stream_kernel", 0), ("bootstrap", 0), ("dense_first", 0), ("fuse_refresh", 0),
                ("two_stage", 0), ("list_fill_pct", 18), ("list_fill_pct", 85), ("gx", 1), ("gx", 16),
                ("cand_budget_mb", 1), ("graph", 0)]


@gpu
@pytest.mark.parametrize("nq,d,store,k", [(1, 768, "f32", 10), (33, 1540, "f16", 10), (65, 768, "bf16", 100),
                                          (129, 1540, "f32", 100), (300, 768, "f16", 10)])
def test_options_do_not_change_the_answer(fo, nq, d, store, k):
    """Each option flipped alone from its default must return (D, I) bit for bit."""
    x = synth(60_000, d, 500 + d)
    q = synth(nq, d, 501 + d)
    e = _engine(x, store)
    xs = _stored(e, x)
    defaults = {"pair": 1, "stream_kernel": 1, "bootstrap": 1, "dense_first": 1, "fuse_refresh": 1,
                "two_stage": 1, "list_fill_pct": 70, "gx": max(1, _sm_count() // 2), "cand_budget_mb": 6 << 10,
                "graph": 1}
    D0, I0 = e.search(q, k)
    s0 = e.stats()
    assert s0["fallback_queries"] == 0 and s0["query_batches"] == 1
    _check_tensor_stats(s0)
    sel = np.arange(nq) if nq <= 64 else np.random.default_rng(nq).choice(nq, 64, replace=False)
    check_topk(D0[sel], I0[sel], q[sel], xs, k, "tensor")
    Do, Io = fo.search(q[sel], xs, k)
    fo.compare_topk(D0[sel], I0[sel], Do, Io, q[sel], xs, rtol=RTOL)
    for name, value in OPTION_FLIPS:
        e.set_option(name, value)
        D, I = e.search(q, k)
        st = e.stats()
        e.set_option(name, defaults[name])
        _check_tensor_stats(st)
        if name == "cand_budget_mb":
            assert st["query_batches"] == -(-nq // 128), st["query_batches"]
        if name == "bootstrap" and s0["sample_rows"] > 0:
            assert st["sample_rows"] == 0
        if st["fallback_queries"] == 0:
            assert np.array_equal(I, I0) and np.array_equal(D, D0), (name, value)
        else:
            check_topk(D[sel], I[sel], q[sel], xs, k, "tensor")
    if nq > 128:
        e.set_option("cand_budget_mb", 1)
        e.search(q, k)
        assert e.stats()["query_batches"] > 1


# ------------------------------------------------------- F. overflow in a later query batch
@gpu
def test_overflowing_query_in_a_later_batch(fo):
    """10,000 copies of one row; query 200 points at it, so its candidate list overflows and the
    query is answered by the exact path.  Every other query scores that row negatively and cannot
    overflow.  With 128-query batches (cand_budget_mb=1) query 200 lies in the second batch: the
    exact path must still answer query 200, not row 72 of its batch."""
    d, k, nq = 768, 100, 300
    x = synth(50_000, d, 601)
    u = x[7000].copy()
    x[7000:17_000] = u
    q = synth(nq, d, 602)
    q[(q @ u) > 0] *= -1
    q[200] = u
    e = _engine(x)
    e.set_option("graph", 0)
    D1, I1 = e.search(q, k)
    s1 = e.stats()
    assert s1["query_batches"] == 1 and s1["fallback_queries"] == 1
    e.set_option("cand_budget_mb", 1)
    D, I = e.search(q, k)
    st = e.stats()
    assert st["query_batches"] == 3 and st["fallback_queries"] == 1
    assert np.array_equal(I[200], np.arange(7000, 7000 + k))
    assert np.array_equal(I, I1) and np.array_equal(D, D1)
    rest = np.r_[np.arange(0, 64), np.arange(128, 200), np.arange(201, 230), np.arange(256, 300)]
    check_topk(D[rest], I[rest], q[rest], x, k, "tensor")
    check_topk(D[200:201], I[200:201], q[200:201], x, k, "exact")
    Do, Io = fo.search(q[rest], x, k)
    fo.compare_topk(D[rest], I[rest], Do, Io, q[rest], x, rtol=RTOL)
