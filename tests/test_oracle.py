"""CPU tests of the oracle (oracle/flatip_oracle.c): pinned against the fp64 brute force, the
committed golden fixture and hand-derived known answers.  The reference has no tests or
golden vectors for this path and faiss is not installable offline ("parity unpinned",
SURVEY.md 8c) -- these are the pins the oracle gets instead."""
import os

import numpy as np
import pytest

from helpers import synth
from oracle import flatip_oracle as fo

FLT_LOWEST = np.finfo(np.float32).min


@pytest.mark.parametrize("use_blas", [True, False])
@pytest.mark.parametrize("n,nq,k,d", [
    (4000, 50, 100, 768),    # blas path, reservoir handler (k >= 100)
    (4000, 7, 10, 768),      # seq path (nq < 20), heap handler
    (3000, 33, 1, 64),       # top-1 handler
    (2500, 25, 99, 96),      # heap handler just below the reservoir switch
    (2500, 19, 100, 96),     # seq path + reservoir
    (9000, 21, 1000, 128),   # large k: several reservoir shrinks
    (5000, 40, 101, 32),
])
def test_oracle_matches_fp64_truth(n, nq, k, d, use_blas):
    x, q = synth(n, d, 1234), synth(nq, d, 4321)
    D, I = fo.search(q, x, k, use_blas=use_blas)
    D64, I64 = fo.brute_force_f64(q, x, k)
    assert D.dtype == np.float32 and I.dtype == np.int64 and D.shape == (nq, k)
    assert (np.diff(D, axis=1) <= 0).all(), "faiss returns rows score-descending"
    fo.compare_topk(D, I, D64.astype(np.float32), I64, q, x, rtol=1e-5)


@pytest.mark.parametrize("n,nq,k,d", [(20000, 64, 100, 768), (6000, 12, 10, 256), (9000, 300, 1000, 128)])
def test_oracle_matches_an_independent_fp32_blas_topk(n, nq, k, d):
    """A second, unrelated fp32 implementation of the same contract -- torch on the CPU: its own
    sgemm (MKL / oneDNN, not the OpenBLAS the restatement calls), the WHOLE score matrix at once
    instead of 4096 x 1024 blocks, `torch.topk` instead of faiss's heap / reservoir handlers --
    must give the restatement's answer up to fp32 ties.  (Not a pin to faiss itself: that needs
    faiss; it guards the blocked handlers of the restatement against a different code path.)"""
    torch = pytest.importorskip("torch")
    x, q = synth(n, d, 31), synth(nq, d, 32)
    x[7000 % n] = x[11]                                   # one exact duplicate
    D, I = fo.search(q, x, k)
    S = torch.from_numpy(q) @ torch.from_numpy(x).T
    top = torch.topk(S, k, dim=1, largest=True, sorted=True)
    fo.compare_topk(D, I, top.values.numpy(), top.indices.numpy().astype(np.int64), q, x, rtol=1e-5)


def test_oracle_unnormalised_fp16_valued():
    x = (synth(3000, 768, 5, normalize=False) * 0.3).astype(np.float16).astype(np.float32)
    q = (synth(30, 768, 6, normalize=False) * 0.3).astype(np.float16).astype(np.float32)
    D, I = fo.search(q, x, 100)
    D64, I64 = fo.brute_force_f64(q, x, 100)
    fo.compare_topk(D, I, D64.astype(np.float32), I64, q, x, rtol=1e-5)


def test_golden_fixture():
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "flatip_small.npz"))
    x, q = g["corpus"].astype(np.float32), g["queries"].astype(np.float32)
    for k in (1, 10, 100):
        D, I = fo.search(q, x, k)
        fo.compare_topk(D, I, g[f"D_k{k}"], g[f"I_k{k}"], q, x, rtol=1e-5)


def test_identity_corpus_known_answer():
    d = 64
    x = np.eye(d, dtype=np.float32)
    q = synth(25, d, 3, normalize=False)
    D, I = fo.search(q, x, 5)
    want = np.argsort(-q, axis=1, kind="stable")[:, :5]
    assert np.array_equal(I, want)
    assert np.array_equal(D, np.take_along_axis(q, want, axis=1))


@pytest.mark.parametrize("nq", [5, 30])          # seq and blas paths
@pytest.mark.parametrize("k", [1, 10, 100])      # top1 / heap / reservoir
def test_fewer_rows_than_k_padding(nq, k):
    x, q = synth(7, 32, 1), synth(nq, 32, 2)
    D, I = fo.search(q, x, k)
    kk = min(k, 7)
    assert (I[:, kk:] == -1).all() and (D[:, kk:] == FLT_LOWEST).all()
    D64, I64 = fo.brute_force_f64(q, x, k)
    assert np.array_equal(I[:, :kk], I64)


@pytest.mark.parametrize("nq", [4, 40])
@pytest.mark.parametrize("k", [1, 20, 150])
def test_all_equal_scores_keep_the_earliest_rows(nq, k):
    """Strict `threshold < score` insertion: once k equal scores are held, later equal rows
    never displace them -> rows 0..k-1 survive (order among ties is implementation-defined)."""
    x = np.tile(synth(1, 48, 9), (1000, 1))
    q = synth(nq, 48, 10)
    D, I = fo.search(q, x, k)
    assert (np.sort(I, axis=1) == np.arange(k)).all()
    assert (D == D[:, :1]).all()


def test_nan_scores_are_never_returned():
    x = synth(50, 16, 1)
    x[7] = np.nan
    q = synth(3, 16, 2)
    D, I = fo.search(q, x, 50)
    assert (I[:, :49] != 7).all() and (I[:, 49] == -1).all() and not np.isnan(D).any()


def test_single_row_and_k1():
    x, q = synth(1, 8, 1), synth(21, 8, 2)
    D, I = fo.search(q, x, 1)
    assert (I == 0).all()
    np.testing.assert_allclose(D[:, 0], q.astype(np.float64) @ x[0].astype(np.float64), rtol=1e-5, atol=1e-7)


def test_compare_topk_rejects_wrong_answers():
    x, q = synth(500, 32, 1), synth(4, 32, 2)
    D, I = fo.brute_force_f64(q, x, 10)
    D = D.astype(np.float32)
    fo.compare_topk(D, I, D, I, q, x)
    bad_I = I.copy()
    bad_I[0, 3] = int(np.setdiff1d(np.arange(500), I[0])[-1])       # a row that is not in the top-k
    with pytest.raises(AssertionError):
        fo.compare_topk(D, bad_I, D, I, q, x)
    bad_D = D.copy()
    bad_D[1, 0] *= 1.001
    with pytest.raises(AssertionError):
        fo.compare_topk(bad_D, I, D, I, q, x)


def test_oracle_indexer_restates_reference_indexer(tmp_path):
    """ids -> str, incremental index_data, [-1] quirk when N < k, file round trip."""
    ix = fo.OracleIndexer(16)
    x = synth(30, 16, 1)
    ix.index_data(list(range(0, 10)), x[:10].astype(np.float16))
    ix.index_data([f"p{i}" for i in range(10, 30)], x[10:])
    res = ix.search_knn(synth(3, 16, 2), 40)
    ids, scores = res[0]
    assert len(res) == 3 and len(ids) == 40 and scores.dtype == np.float32
    assert all(isinstance(i, str) for i in ids)
    assert ids[30:] == ["p29"] * 10          # index_id_to_db_id[-1], reference src/index.py:44
    ix.serialize(str(tmp_path))
    iy = fo.OracleIndexer(16)
    iy.deserialize_from(str(tmp_path))
    assert iy.index_id_to_db_id == ix.index_id_to_db_id and np.array_equal(iy.rows, ix.rows)
    assert os.path.getsize(tmp_path / "index.faiss") == 45 + 4 * 30 * 16


# ------------------------------------------------------------------------------------------
# Pins that activate the day `import faiss` works (faiss-cpu==1.8.0, reference environment.yml:138):
# the restatement, the index.faiss writer / reader and the drop-in's host logic against the REAL
# library.  Skipped where faiss is not installed.
# ------------------------------------------------------------------------------------------
def test_oracle_backend_is_reported():
    """Without faiss the oracle says it is a port; with faiss it must say it is the reference."""
    assert fo.backend_kind() == ("reference" if fo.real_faiss() is not None else "port")
    assert ("faiss" in fo.backend_description())


@pytest.mark.parametrize("n,nq,k,d", [(4000, 50, 100, 768), (4000, 7, 10, 768), (3000, 33, 1, 64),
                                      (9000, 21, 1000, 128), (50, 5, 100, 32)])
def test_restatement_matches_real_faiss(n, nq, k, d):
    faiss = pytest.importorskip("faiss")
    x, q = synth(n, d, 1234), synth(nq, d, 4321)
    index = faiss.IndexFlatIP(d)
    index.add(x)
    Df, If = index.search(q, k)
    Dr, Ir = fo.restatement_search(q, x, k)
    assert np.array_equal(If >= 0, Ir >= 0), "padding pattern (ntotal < k)"
    fo.compare_topk(Dr, Ir, Df, If, q, x, rtol=1e-5)
    assert np.array_equal(Df[If < 0], Dr[Ir < 0])            # -FLT_MAX padding scores


def test_index_faiss_files_are_interchangeable_with_real_faiss(tmp_path):
    faiss = pytest.importorskip("faiss")
    rows = synth(1000, 24, 3)
    ours, theirs = str(tmp_path / "ours.faiss"), str(tmp_path / "theirs.faiss")
    fo.write_index_flat_ip(ours, rows)
    index = faiss.IndexFlatIP(24)
    index.add(rows)
    faiss.write_index(index, theirs)
    assert open(ours, "rb").read() == open(theirs, "rb").read(), "IxFI byte layout"
    back = faiss.read_index(ours)
    assert back.ntotal == 1000 and back.d == 24 and back.metric_type == faiss.METRIC_INNER_PRODUCT
    assert np.array_equal(fo.read_index_flat_ip(theirs), rows)
    import b2ip
    d, n, blocks = b2ip.stream_flat_ip_rows(theirs)
    assert (d, n) == (24, 1000) and np.array_equal(np.concatenate(list(blocks)), rows)
