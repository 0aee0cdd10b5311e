"""`MultiGpuEngine`: the row-sharded search of `ShardedIndex`, driven from ONE process.

The reference runs its retrieval in a single process (passage_retrieval.py never initialises
torch.distributed, SURVEY.md 1), so a drop-in `Indexer` cannot assume `torchrun`.  This class
gives that single process every GPU of the box: one `Engine` (= one C-ABI handle, one row
shard) per device, host threads that run the per-device searches concurrently (the ctypes call
releases the GIL) and the SAME fused peer-direct exchange as the one-process-per-GPU path
(`b2ip_search_exchange`: global threshold round, every finalize kernel stores its block into
the owner GPU's gather buffer over NVLink, each GPU merges the queries it owns) -- between
handles of one process the peer buffers are plain device pointers.  Each GPU then copies its
slice of the result to the host on its own copy engine.  Without P2P between the devices the
per-shard results are copied to the first device and merged there (`b2ip_merge_topk_strided`).  Same surface as
`Engine` (add / search / ntotal / export_rows / reserve / stats / close), same results: the
merge keeps score-descending order and the lower GLOBAL row among equal scores.

Every `add` cuts its rows into consecutive slices that level the shards' running totals, so
shards stay balanced however the caller chunks its data; a per-engine segment table maps
local rows back to global ids.
"""
from __future__ import annotations

import bisect
import os
from concurrent.futures import ThreadPoolExecutor
from typing import List, Optional, Sequence, Tuple

import numpy as np

from .engine import Engine, merge_topk


class SegmentMap:
    """Local row -> global row for one shard: segments (local_start, global_start, n) appended
    in increasing global order."""

    def __init__(self):
        self.segments: List[Tuple[int, int, int]] = []
        self.n_local = 0
        self._cache = None

    def append(self, global_start: int, n: int) -> None:
        if n <= 0:
            return
        if self.segments and global_start < self.segments[-1][1] + self.segments[-1][2]:
            raise ValueError("segments must be appended in increasing global row order")
        if self.segments and self.segments[-1][1] + self.segments[-1][2] == global_start:
            ls, gs, m = self.segments[-1]
            self.segments[-1] = (ls, gs, m + n)
        else:
            self.segments.append((self.n_local, int(global_start), int(n)))
        self.n_local += n
        self._cache = None

    def single_offset(self) -> Optional[int]:
        """global - local when the shard is one contiguous segment (the engine can add it)."""
        if len(self.segments) == 1:
            return self.segments[0][1] - self.segments[0][0]
        return None

    def to_global(self, rows_local):
        """torch int64 tensor of local rows (-1 = padding) -> global rows."""
        import torch
        if not self.segments:
            return rows_local
        if self._cache is None or self._cache[0].device != rows_local.device:
            ls = torch.tensor([s[0] for s in self.segments], dtype=torch.int64, device=rows_local.device)
            delta = torch.tensor([s[1] - s[0] for s in self.segments], dtype=torch.int64,
                                 device=rows_local.device)
            self._cache = (ls, delta)
        ls, delta = self._cache
        seg = torch.bucketize(rows_local.clamp(min=0), ls, right=True) - 1
        return torch.where(rows_local >= 0, rows_local + delta[seg], rows_local)

    def local_mask(self, allowed):
        """The shard's slice of a global allowed-row mask (numpy or torch bool, one entry per
        global row), in local row order: the shard's segments are interleaved with the other
        shards', so this is one slice per segment."""
        parts = [allowed[gs:gs + n] for _, gs, n in self.segments]
        if type(allowed).__module__.startswith("torch"):
            import torch
            return torch.cat(parts) if parts else allowed[:0]
        return np.concatenate(parts) if parts else allowed[:0]

    def overlaps(self, g0: int, g1: int):
        """(local_start, global_start, n) pieces of this shard inside global rows [g0, g1)."""
        starts = [s[1] for s in self.segments]
        i = max(0, bisect.bisect_right(starts, g0) - 1)
        for ls, gs, n in self.segments[i:]:
            if gs >= g1:
                break
            a, b = max(gs, g0), min(gs + n, g1)
            if a < b:
                yield ls + (a - gs), a, b - a


def level_split(totals: Sequence[int], n: int) -> List[int]:
    """How many of n new rows each shard takes (consecutive slices, in shard order) so that the
    running totals stay level: shard g aims at its share of the new grand total; totals never
    differ by more than one row once they were level."""
    G, N, left, out = len(totals), sum(totals) + n, n, []
    for g in range(G):
        target = N * (g + 1) // G - N * g // G
        take = min(max(target - totals[g], 0), left)
        out.append(take)
        left -= take
    assert left == 0, (totals, n, out)
    return out


def merge_range_results(parts):
    """Merge per-shard range search answers [(lims [nq+1], D [total], I [total]), ...] (global
    rows, ascending per query) into one: per query, the union of the shards' hits in ascending row
    order.  Shards hold interleaved row segments, so this is a per-query merge, not a concatenation."""
    parts = [(np.asarray(l, np.int64), np.asarray(d, np.float32), np.asarray(i, np.int64)) for l, d, i in parts]
    nq = len(parts[0][0]) - 1
    qs = [np.repeat(np.arange(nq, dtype=np.int64), np.diff(l)) for l, _, _ in parts]
    q = np.concatenate(qs)
    D = np.concatenate([d[:l[-1]] for l, d, _ in parts])
    I = np.concatenate([i[:l[-1]] for l, _, i in parts])
    order = np.lexsort((I, q))
    lims = np.zeros(nq + 1, dtype=np.int64)
    np.cumsum(np.bincount(q, minlength=nq), out=lims[1:])
    return lims, D[order], I[order]


class MultiGpuEngine:
    def __init__(self, d: int, devices: Optional[Sequence[int]] = None, store: str = "f32",
                 shadow: Optional[str] = None):
        import torch
        if devices is None:
            devices = list(range(torch.cuda.device_count()))
        devices = [int(x) for x in devices]
        if not devices:
            raise RuntimeError("MultiGpuEngine needs at least one CUDA device (no CPU fallback)")
        self._torch = torch
        self.d, self.store, self.devices = int(d), store, devices
        self.engines = [Engine(d, dev, store=store, shadow=shadow) for dev in devices]
        self.maps = [SegmentMap() for _ in devices]
        self._n = 0
        self._pool = ThreadPoolExecutor(max_workers=len(devices))
        self._last_stats: List[dict] = []
        self._x_ok = None if os.environ.get("B2IP_PEER_EXCHANGE", "1") != "0" else False
        self._x_ex, self._x_bufs, self._x_slot, self._x_thr_cap, self._x_seq = None, None, 0, 0, 0
        self.exchange_searches = 0
        self._group, self._group_ok = None, (None if os.environ.get("B2IP_PEER_EXCHANGE", "1") != "0" else False)

    # -- lifetime / configuration ----------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_group", None) is not None:
            from ._lib import load
            load().b2ip_group_destroy(self._group)
            self._group = None
        for e in getattr(self, "engines", []):
            e.close()
        if getattr(self, "_pool", None) is not None:
            self._pool.shutdown(wait=False)
            self._pool = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def device(self) -> int:
        return self.devices[0]

    @property
    def ntotal(self) -> int:
        return self._n

    def reserve(self, n_rows: int) -> None:
        per = -(-int(n_rows) // len(self.engines))
        for e in self.engines:
            e.reserve(per + len(self.engines))

    def set_option(self, name: str, value: int) -> None:
        for e in self.engines:
            e.set_option(name, value)

    # -- data ------------------------------------------------------------------------
    def add(self, rows) -> None:
        """Rows get global ids ntotal .. ntotal+n-1.  The chunk is cut into consecutive slices,
        one per device, sized to LEVEL the shards' running totals (a remainder or a chunk smaller
        than the number of devices goes to the least-filled shards, not always to device 0)."""
        n = int(rows.shape[0])
        jobs, lo = [], 0
        for g, take in enumerate(level_split([m.n_local for m in self.maps], n)):
            hi = lo + take
            if hi > lo:
                self.maps[g].append(self._n + lo, hi - lo)
                jobs.append(self._pool.submit(self._add_one, g, rows[lo:hi]))
            lo = hi
        assert lo == n
        for j in jobs:
            j.result()
        for g, e in enumerate(self.engines):
            e.set_row_segments(self.maps[g].segments)      # the engine reports global ids itself
        self._n += n

    def _add_one(self, g: int, part) -> None:
        torch = self._torch
        if type(part).__module__.startswith("torch") and part.is_cuda and part.device.index != self.devices[g]:
            part = part.to(torch.device("cuda", self.devices[g]))
        with torch.cuda.device(self.devices[g]):
            self.engines[g].add(part)

    def export_rows(self, row0: int, n: int) -> np.ndarray:
        out = np.empty((n, self.d), dtype=np.float32)
        for g, e in enumerate(self.engines):
            for ls, gs, m in self.maps[g].overlaps(row0, row0 + n):
                out[gs - row0:gs - row0 + m] = e.export_rows(ls, m)
        return out

    # -- search ----------------------------------------------------------------------
    def _search_one(self, g: int, q_dev0, k: int, mode: str, allowed=None):
        torch = self._torch
        dev = torch.device("cuda", self.devices[g])
        with torch.cuda.device(dev):
            q = q_dev0 if q_dev0.device == dev else q_dev0.to(dev)      # fan-out over NVLink
            if allowed is None:
                D, I = self.engines[g].search(q, k, mode=mode)
            else:
                mask = self.maps[g].local_mask(allowed)
                if type(mask).__module__.startswith("torch") and mask.device != dev:
                    mask = mask.to(dev)
                D, I = self.engines[g].search(q, k, mode=mode, allowed=mask)
            st = self.engines[g].stats()
            torch.cuda.current_stream(dev).synchronize()
        return D, I, st

    FLAG_BYTES = 256

    def _exchange(self, nq: int, k: int):
        """Per-device gather / threshold / flag buffers of the fused exchange (two parities) and
        the b2ip_exchange_t of every device; None when the devices cannot reach each other."""
        if self._x_ok is False:
            return None
        need = (nq * k * 12 + 15) // 16 * 16
        if self._x_ex is not None and need <= self._x_slot and nq <= self._x_thr_cap:
            return self._x_ex
        from ._lib import GATHER_OWNER, B2ipError, Exchange
        torch = self._torch
        G = len(self.engines)
        if self._x_ok is None and len(set(self.devices)) != len(self.devices):
            # shards that share a GPU cannot wait for each other inside kernels (the waiting CTAs
            # could keep the peer's kernels off the SMs): copy-and-merge path
            self._x_ok = False
            return None
        if self._x_ok is None:
            try:
                for a in range(G):
                    for b in range(G):
                        self.engines[a].enable_peer_access(self.devices[b])
                self._x_ok = True
            except B2ipError:
                self._x_ok = False
                return None
        slot = max(1 << 16, (need + need // 4 + 65535) // 65536 * 65536, self._x_slot)
        thr_cap = max((nq + nq // 4 + 1023) // 1024 * 1024, self._x_thr_cap)
        thr_bytes = G * thr_cap * 4
        total = 2 * G * slot + 2 * thr_bytes + 2 * self.FLAG_BYTES
        for dev in self.devices:
            torch.cuda.synchronize(dev)
        bufs = [torch.zeros(total, dtype=torch.uint8, device=torch.device("cuda", dev)) for dev in self.devices]
        for dev in self.devices:
            torch.cuda.synchronize(dev)
        ptrs = [b.data_ptr() for b in bufs]
        exs = []
        for g in range(G):
            pair = []
            for parity in (0, 1):
                ex = Exchange()
                ex.world, ex.rank, ex.slot_bytes = G, g, slot
                ex.thr_stride, ex.gather_mode = thr_cap, GATHER_OWNER
                for p in range(G):
                    ex.gather[p] = ptrs[p] + parity * G * slot
                    ex.gthr[p] = ptrs[p] + 2 * G * slot + parity * thr_bytes
                    ex.flags[p] = ptrs[p] + 2 * G * slot + 2 * thr_bytes + parity * self.FLAG_BYTES
                pair.append(ex)
            exs.append(pair)
        self._x_bufs, self._x_slot, self._x_thr_cap, self._x_ex, self._x_seq = bufs, slot, thr_cap, exs, 0
        return exs

    def _group_search(self, q_host: np.ndarray, k: int, host_out):
        """b2ip_group_search over this engine's handles.  Returns the exchange status (0 = done,
        > 0 = a candidate list overflowed: repeat shard by shard) or None when the devices cannot
        reach each other (the group cannot be created)."""
        import ctypes
        from ._lib import B2IP_F16, B2IP_F32, B2ipError, load
        lib = load()
        if self._group is None:
            arr = (ctypes.c_void_p * len(self.engines))(*[e._h.value for e in self.engines])
            grp = ctypes.c_void_p()
            rc = lib.b2ip_group_create(len(self.engines), arr, ctypes.byref(grp))
            if rc != 0:
                self._group_ok = False
                return None
            self._group, self._group_ok = grp, True
        status = ctypes.c_int64(0)
        D, I = host_out
        assert D.flags["C_CONTIGUOUS"] and I.flags["C_CONTIGUOUS"] and D.dtype == np.float32 and I.dtype == np.int64
        rc = lib.b2ip_group_search(self._group, q_host.shape[0], ctypes.c_void_p(q_host.ctypes.data),
                                   B2IP_F16 if q_host.dtype == np.float16 else B2IP_F32, int(k),
                                   ctypes.c_void_p(D.ctypes.data), ctypes.c_void_p(I.ctypes.data),
                                   ctypes.byref(status))
        if rc != 0:
            msg = lib.b2ip_group_last_error(self._group)
            raise B2ipError(rc, msg.decode() if msg else "")
        return int(status.value)

    def _search_exchange_one(self, g: int, q_dev0, k: int, ex, seq: int, host_out, lo: int, hi: int):
        """Device g: fan-in of the queries, search + exchange + merge of the queries it owns, and
        (host output) the D2H of that slice on this device's copy engine."""
        torch = self._torch
        dev = torch.device("cuda", self.devices[g])
        with torch.cuda.device(dev):
            q = q_dev0 if q_dev0.device == dev else q_dev0.to(dev)
            D, I, status = self.engines[g].search_exchange(q, k, ex, seq)
            st = self.engines[g].stats()
            if status == 0 and host_out is not None and hi > lo:
                self.engines[g].download(D, host_out[0][lo:hi])
                self.engines[g].download(I, host_out[1][lo:hi])
        return D, I, st, status

    def search(self, queries, k: int, mode: str = "auto", out=None, allowed=None):
        """numpy in -> numpy out, torch CUDA tensor in -> tensors on the first device.  `allowed`
        (bool per global row, numpy or torch) restricts the search as in `Engine.search`: each
        shard searches its own slice of the mask and the per-shard results are merged."""
        torch = self._torch
        k = int(k)
        G = len(self.engines)
        dev0 = torch.device("cuda", self.devices[0])
        is_t = type(queries).__module__.startswith("torch")
        if is_t:
            q_dev0 = queries if queries.dtype in (torch.float16, torch.float32) else queries.float()
            q_dev0 = q_dev0.contiguous()
            torch.cuda.current_stream(q_dev0.device).synchronize()
            nq = q_dev0.shape[0]
        else:
            q_host = np.asarray(queries)
            if q_host.dtype not in (np.float16, np.float32):
                q_host = q_host.astype(np.float32)
            q_host = np.ascontiguousarray(q_host)
            if q_host.ndim != 2 or q_host.shape[1] != self.d:
                raise ValueError(f"expected [nq,{self.d}] queries, got {q_host.shape}")
            nq = q_host.shape[0]
            with torch.cuda.device(dev0):
                # one staged upload (pinned double buffering inside the library), then P2P fan-out;
                # float16 queries stay float16 until they are on the device
                q_dev0 = torch.empty((nq, self.d), device=dev0,
                                     dtype=torch.float16 if q_host.dtype == np.float16 else torch.float32)
                if nq:
                    self.engines[0].upload(q_dev0, q_host)
        host_out = None
        if not is_t:
            host_out = out if out is not None else (np.empty((nq, k), np.float32), np.empty((nq, k), np.int64))
        if nq == 0:
            if is_t:
                return (torch.empty((0, k), dtype=torch.float32, device=dev0),
                        torch.empty((0, k), dtype=torch.int64, device=dev0))
            return host_out
        D = I = None
        if allowed is not None and len(allowed) != self._n:
            raise ValueError(f"allowed has {len(allowed)} entries, the index holds {self._n} rows")
        filtered = allowed is not None           # the fused exchange paths take no filter
        if not is_t and G > 1 and mode != "exact" and self._group_ok is not False and not filtered:
            # host queries: ONE native call runs uploads, searches + fused exchange and downloads
            # of all GPUs on the library's own worker threads (b2ip_group_search)
            status = self._group_search(q_host, k, host_out)
            if status == 0:
                self.exchange_searches += 1
                self._last_stats = [e.stats() for e in self.engines]
                return host_out
            if status is None:                       # no P2P path between the devices
                pass
        ex = self._exchange(nq, k) if (G > 1 and mode != "exact" and is_t and not filtered) else None
        if ex is not None:
            self._x_seq += 1
            per = -(-nq // G)
            spans = [(min(g * per, nq), min(min(g * per, nq) + per, nq)) for g in range(G)]
            parts = [self._pool.submit(self._search_exchange_one, g, q_dev0, k, ex[g][self._x_seq & 1],
                                       self._x_seq, host_out, *spans[g]) for g in range(G)]
            res = [p.result() for p in parts]
            self._last_stats = [r[2] for r in res]
            if all(r[3] == 0 for r in res):
                self.exchange_searches += 1
                if not is_t:
                    return host_out
                with torch.cuda.device(dev0):
                    return (torch.cat([r[0].to(dev0) for r in res]), torch.cat([r[1].to(dev0) for r in res]))
            # a candidate list overflowed somewhere (same status on every device): repeat below
        parts = [self._pool.submit(self._search_one, g, q_dev0, k, mode, allowed) for g in range(G)]
        res = [p.result() for p in parts]
        self._last_stats = [r[2] for r in res]
        with torch.cuda.device(dev0):
            if len(res) == 1:
                D, I = res[0][0], res[0][1]
            else:
                gD = torch.empty((G, nq, k), dtype=torch.float32, device=dev0)
                gI = torch.empty((G, nq, k), dtype=torch.int64, device=dev0)
                for g, r in enumerate(res):                 # one P2P copy per shard, straight into place
                    gD[g].copy_(r[0])
                    gI[g].copy_(r[1])
                D, I = merge_topk(gD, gI, k)
        if is_t:
            return D, I
        self.engines[0].download(D.contiguous(), host_out[0])
        self.engines[0].download(I.contiguous(), host_out[1])
        return host_out

    def _range_one(self, g: int, queries, radius: float, mode: str):
        torch = self._torch
        dev = torch.device("cuda", self.devices[g])
        with torch.cuda.device(dev):
            q = queries
            if type(q).__module__.startswith("torch") and q.device != dev:
                q = q.to(dev)
            lims, D, I = self.engines[g].range_search(q, radius, mode=mode)
            if type(lims).__module__.startswith("torch"):
                lims, D, I = lims.cpu().numpy(), D.cpu().numpy(), I.cpu().numpy()
            st = self.engines[g].stats()
        return (lims, D, I), st

    def range_search(self, queries, radius: float, mode: str = "auto"):
        """One range search per shard, merged per query by global row (`merge_range_results`).
        numpy in -> numpy out; torch CUDA tensor in -> CUDA tensors on the first device."""
        torch = self._torch
        is_t = type(queries).__module__.startswith("torch")
        if is_t:
            queries = queries.contiguous()
            torch.cuda.current_stream(queries.device).synchronize()
        jobs = [self._pool.submit(self._range_one, g, queries, radius, mode) for g in range(len(self.engines))]
        res = [j.result() for j in jobs]
        self._last_stats = [r[1] for r in res]
        lims, D, I = merge_range_results([r[0] for r in res])
        if is_t:
            dev0 = torch.device("cuda", self.devices[0])
            return (torch.from_numpy(lims).to(dev0), torch.from_numpy(D).to(dev0), torch.from_numpy(I).to(dev0))
        return lims, D, I

    def download(self, src, dst: np.ndarray) -> None:
        """dst (host array) <- src (CUDA tensor on any of this engine's devices)."""
        g = self.devices.index(src.device.index)
        with self._torch.cuda.device(src.device):
            self.engines[g].download(src, dst)

    def stats(self) -> dict:
        """Per-device stats of the last search, plus sums of the additive counters."""
        if not self._last_stats:
            return {}
        agg = dict(self._last_stats[0])
        for key in ("coarse_launches", "total_launches", "coarse_flops", "candidates", "rescored",
                    "fallback_queries"):
            agg[key] = sum(s[key] for s in self._last_stats)
        for key in ("coarse_ms", "total_ms", "refresh_ms", "finalize_ms"):
            agg[key] = max(s[key] for s in self._last_stats)
        agg["ntotal"] = self._n
        agg["per_device"] = self._last_stats
        return agg
