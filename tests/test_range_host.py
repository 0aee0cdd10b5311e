"""Range search pieces that need no GPU: the per-query merge of shard answers, the ordering and id
mapping of `Indexer.search_range`, and the C ABI declarations of the two range functions."""
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _random_answer(rng, nq, rows, p):
    """CSR answer over the given global rows: each (query, row) kept with probability p."""
    keep = rng.random((nq, len(rows))) < p
    lims = np.zeros(nq + 1, np.int64)
    lims[1:] = np.cumsum(keep.sum(axis=1))
    I = np.concatenate([rows[k] for k in keep]).astype(np.int64) if nq else np.zeros(0, np.int64)
    D = rng.standard_normal(len(I)).astype(np.float32)
    return lims, D, I


@pytest.mark.parametrize("seed", range(6))
def test_merge_range_results_matches_a_reference(seed):
    from b2ip.multi import merge_range_results
    rng = np.random.default_rng(seed)
    nq, n, G = int(rng.integers(0, 9)), int(rng.integers(1, 400)), int(rng.integers(1, 5))
    # interleaved segments of random length, dealt to the shards in turn
    owner = np.repeat(np.arange(1000) % G, rng.integers(1, 30, size=1000))[:n]
    parts = []
    for g in range(G):
        rows = np.nonzero(owner == g)[0]
        parts.append(_random_answer(rng, nq, rows, p=0 if g == 1 else rng.random()))
    lims, D, I = merge_range_results(parts)
    assert lims.dtype == np.int64 and D.dtype == np.float32 and I.dtype == np.int64
    assert lims.shape == (nq + 1,) and lims[0] == 0 and len(D) == len(I) == lims[-1]
    for q in range(nq):
        ref = {}
        for pl, pD, pI in parts:
            for j in range(pl[q], pl[q + 1]):
                ref[int(pI[j])] = pD[j]
        rows = sorted(ref)
        assert I[lims[q]:lims[q + 1]].tolist() == rows
        assert np.array_equal(D[lims[q]:lims[q + 1]], np.array([ref[r] for r in rows], np.float32))


def test_merge_range_results_of_empty_parts():
    from b2ip.multi import merge_range_results
    empty = (np.zeros(4, np.int64), np.zeros(0, np.float32), np.zeros(0, np.int64))
    lims, D, I = merge_range_results([empty, empty])
    assert lims.tolist() == [0, 0, 0, 0] and len(D) == 0 and len(I) == 0
    lims, D, I = merge_range_results([(np.zeros(1, np.int64), np.zeros(0, np.float32), np.zeros(0, np.int64))])
    assert lims.tolist() == [0] and len(D) == 0


class _FakeEngine:
    """Stands in for Engine: a fixed CSR answer, rows ascending per query as the library returns them."""
    d, store, device = 4, "f32", 0

    def __init__(self, answer):
        self.answer = answer
        self.calls = []

    def range_search(self, q, radius, mode="auto"):
        self.calls.append((np.asarray(q).shape, np.asarray(q).dtype, radius))
        return self.answer


def test_search_range_orders_by_score_and_maps_ids():
    from b2ip.indexer import Indexer
    lims = np.array([0, 4, 4, 7], np.int64)
    I = np.array([0, 2, 5, 9, 1, 3, 8], np.int64)
    D = np.array([0.5, 0.9, 0.5, -1.0, 2.0, 2.0, 3.0], np.float32)
    eng = _FakeEngine((lims, D, I))
    idx = Indexer.from_engine(eng, ids=[f"doc{i}" for i in range(10)])
    out = idx.search_range(np.zeros((3, 4), np.float16), 0.25)
    assert eng.calls == [((3, 4), np.float16, 0.25)]
    assert len(out) == 3
    ids, scores = out[0]
    assert ids == ["doc2", "doc0", "doc5", "doc9"]          # score descending, ties to the lower row
    assert scores.dtype == np.float32 and scores.tolist() == [np.float32(0.9), 0.5, 0.5, -1.0]
    assert out[1][0] == [] and len(out[1][1]) == 0
    assert out[2][0] == ["doc8", "doc1", "doc3"] and out[2][1].tolist() == [3.0, 2.0, 2.0]
    assert idx.search_range(np.zeros((0, 4), np.float32), 0.0) == []


def test_search_range_converts_other_dtypes_to_float32():
    from b2ip.indexer import Indexer
    eng = _FakeEngine((np.zeros(2, np.int64), np.zeros(0, np.float32), np.zeros(0, np.int64)))
    idx = Indexer.from_engine(eng, ids=[])
    assert idx.search_range(np.zeros((1, 4), np.float64), 1.0) == [([], pytest.approx(np.zeros(0)))]
    assert eng.calls[0][1] == np.float32


def test_range_functions_are_declared_in_plain_c():
    import b2ip
    hdr = os.path.join(ROOT, "include", "b2ip.h")
    out = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-fsyntax-only", "-x", "c", hdr],
                         capture_output=True, text=True)
    assert out.returncode == 0 and not out.stderr.strip(), out.stderr
    text = re.sub(r"/\*.*?\*/", "", open(hdr).read(), flags=re.S)
    for name in ("b2ip_range_search", "b2ip_range_fetch"):
        assert re.search(r"\bint " + name + r"\s*\(", text), name
        assert name in b2ip.SYMBOLS
    if os.path.exists(b2ip.LIB_PATH):
        syms = subprocess.run(["nm", "-D", "--defined-only", b2ip.LIB_PATH], capture_output=True, text=True).stdout
        exported = set(re.findall(r" T (b2ip_[a-z_0-9]+)", syms))
        assert {"b2ip_range_search", "b2ip_range_fetch"} <= exported
