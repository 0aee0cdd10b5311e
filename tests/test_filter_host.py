"""Filtered search pieces that need no GPU: packing an allowed-row mask into the bitmap the library
reads, cutting a global mask into each shard's local mask, the `allowed_ids` -> mask conversion
and padding trim of `Indexer.search_knn`, and the C declaration of b2ip_search_filtered."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLT_MAX = float(np.finfo(np.float32).max)


def _bits_of(words, n):
    words = np.asarray(words).view(np.uint32)
    return np.array([(int(words[r >> 5]) >> (r & 31)) & 1 for r in range(n)], dtype=bool)


@pytest.mark.parametrize("n", [1, 31, 32, 33, 1000])
@pytest.mark.parametrize("kind", ["numpy", "torch"])
def test_pack_allowed(n, kind):
    from b2ip.engine import pack_allowed
    rng = np.random.default_rng(n)
    for mask in (rng.random(n) < 0.5, np.ones(n, bool), np.zeros(n, bool)):
        if kind == "torch":
            import torch
            words = pack_allowed(torch.from_numpy(mask))
            assert words.dtype == torch.int32 and words.device.type == "cpu"
            words = words.numpy()
        else:
            words = pack_allowed(mask)
            assert words.dtype == np.dtype("<u4")
        assert words.shape == (-(-n // 32),)
        assert np.array_equal(_bits_of(words, n), mask)
        # bits past n in the last word stay clear
        assert np.array_equal(_bits_of(words, len(words) * 32)[n:], np.zeros(len(words) * 32 - n, bool))
        ref = np.packbits(mask, bitorder="little")
        assert np.array_equal(words.view(np.uint8)[:len(ref)], ref)


def test_pack_allowed_rejects_other_masks():
    from b2ip.engine import pack_allowed
    with pytest.raises(ValueError):
        pack_allowed(np.ones(5, np.int32))
    with pytest.raises(ValueError):
        pack_allowed(np.ones((2, 5), bool))


@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("kind", ["numpy", "torch"])
def test_local_masks_follow_interleaved_segments(seed, kind):
    """MultiGpuEngine.add levels the shards chunk by chunk, so every shard holds interleaved
    segments of the global rows; each shard's mask lists its rows in local order."""
    from b2ip.multi import SegmentMap, level_split
    rng = np.random.default_rng(seed)
    G = int(rng.integers(2, 5))
    maps = [SegmentMap() for _ in range(G)]
    owner, local = [], []          # per global row: shard and local row, as add() assigns them
    total = 0
    for _ in range(int(rng.integers(1, 8))):
        n = int(rng.integers(0, 300))
        lo = 0
        for g, take in enumerate(level_split([m.n_local for m in maps], n)):
            maps[g].append(total + lo, take)
            owner += [g] * take
            local += list(range(maps[g].n_local - take, maps[g].n_local))
            lo += take
        total += n
    owner, local = np.array(owner, int), np.array(local, int)
    mask = rng.random(total) < 0.4
    for g in range(G):
        want = np.zeros(maps[g].n_local, bool)
        want[local[owner == g]] = mask[owner == g]
        got = maps[g].local_mask(mask if kind == "numpy" else __import__("torch").from_numpy(mask))
        got = np.asarray(got)
        assert got.dtype == bool and np.array_equal(got, want), g


class _FakeEngine:
    """Stands in for Engine: records the mask of each search and returns a fixed answer."""
    d, store, device = 4, "f32", 0

    def __init__(self, n, answer=None):
        self.n = n
        self.answer = answer
        self.masks = []

    @property
    def ntotal(self):
        return self.n

    def add(self, rows):
        self.n += len(rows)

    def search(self, q, k, mode="auto", allowed=None):
        self.masks.append(None if allowed is None else np.asarray(allowed).copy())
        return self.answer


def test_allowed_ids_to_mask():
    from b2ip.indexer import Indexer
    ids = ["a", "b", 7, "c", "b", "7", "d"]
    idx = Indexer.from_engine(_FakeEngine(len(ids)), ids=ids)
    # duplicated ids: every row; ids match as str (7 and "7"); unknown ids are ignored
    m = idx.allowed_mask(["b", "7", "zz", "b", 12345])
    assert m.tolist() == [False, True, True, False, True, True, False]
    assert not idx.allowed_mask([]).any() and not idx.allowed_mask(["nope"]).any()
    assert idx.allowed_mask(iter(["a", "d"])).tolist() == [True, False, False, False, False, False, True]
    lookup = idx._id_rows
    idx.allowed_mask(["c"])
    assert idx._id_rows is lookup                 # built once, then reused
    # index_data appends ids: the lookup is rebuilt with them
    idx.index_data(["e", "a"], np.zeros((2, 4), np.float32))
    assert idx._id_rows is None
    assert idx.allowed_mask(["a", "e"]).tolist() == [True] + [False] * 6 + [True, True]


def test_search_knn_with_allowed_ids_drops_the_padding():
    from b2ip.indexer import Indexer
    ids = [f"doc{i}" for i in range(6)]
    D = np.array([[0.9, 0.5, -FLT_MAX], [-FLT_MAX] * 3], np.float32)
    I = np.array([[4, 1, -1], [-1, -1, -1]], np.int64)
    eng = _FakeEngine(6, (D, I))
    idx = Indexer.from_engine(eng, ids=ids)
    out = idx.search_knn(np.zeros((2, 4), np.float32), 3, allowed_ids=["doc1", "doc4", "other"])
    assert eng.masks[-1].tolist() == [False, True, False, False, True, False]
    assert out[0][0] == ["doc4", "doc1"] and out[0][1].tolist() == [np.float32(0.9), np.float32(0.5)]
    assert out[1][0] == [] and len(out[1][1]) == 0
    # without a filter: today's answer, padding mapped like the reference (ids[-1])
    out = idx.search_knn(np.zeros((2, 4), np.float32), 3)
    assert eng.masks[-1] is None
    assert out[0][0] == ["doc4", "doc1", "doc5"] and len(out[0][1]) == 3


def test_search_knn_with_allowed_ids_on_an_empty_index():
    from b2ip.indexer import Indexer
    idx = Indexer.from_engine(_FakeEngine(0), ids=[])
    out = idx.search_knn(np.zeros((3, 4), np.float32), 5, allowed_ids=["x"])
    assert len(out) == 3 and all(i == [] and len(s) == 0 for i, s in out)


def test_search_filtered_declaration_matches_the_header():
    import b2ip
    from b2ip import _lib
    hdr = os.path.join(ROOT, "include", "b2ip.h")
    out = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-fsyntax-only", "-x", "c", hdr],
                         capture_output=True, text=True)
    assert out.returncode == 0 and not out.stderr.strip(), out.stderr
    text = re.sub(r"/\*.*?\*/", "", open(hdr).read(), flags=re.S)
    m = re.search(r"\bint b2ip_search_filtered\s*\(([^)]*)\)", text)
    assert m, "b2ip_search_filtered is not declared"
    c_types = [re.sub(r"\s+", " ", re.sub(r"\w+$", "", a.strip())).strip() for a in m.group(1).split(",")]
    to_ctypes = {"b2ip_handle": ctypes.c_void_p, "int64_t": ctypes.c_int64, "const void*": ctypes.c_void_p,
                 "int": ctypes.c_int, "const uint32_t*": ctypes.c_void_p, "float*": ctypes.c_void_p,
                 "int64_t*": ctypes.c_void_p}
    want = [to_ctypes[t] for t in c_types]
    assert len(want) == 11
    assert "b2ip_search_filtered" in b2ip.SYMBOLS
    if os.path.exists(b2ip.LIB_PATH):
        lib = _lib.load()
        assert list(lib.b2ip_search_filtered.argtypes) == want
        assert lib.b2ip_search_filtered.restype == ctypes.c_int
