"""`Engine`: one row shard of the exact IP index on one B200, over the C ABI.

Accepts numpy arrays (host buffers) or torch CUDA tensors (device buffers, zero copy); torch is
only imported when a tensor is handed in.  Mirrors what the reference does with its faiss
object in src/index.py: `add` <- index.add (:30), `search` <- index.search (:42),
`ntotal` <- index.ntotal (:67), `export_rows` <- what faiss.write_index reads (:53).
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import numpy as np

from . import _lib
from ._lib import (B2IP_BF16, B2IP_F16, B2IP_F32, MEM_DEVICE, MEM_HOST, MODE_AUTO, MODE_EXACT,
                   MODE_TENSOR, STORE_BF16, STORE_F16, STORE_F32, B2ipError, Stats, check)

_MODES = {"auto": MODE_AUTO, "tensor": MODE_TENSOR, "exact": MODE_EXACT}


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


def pack_allowed(allowed):
    """Allowed-row mask (bool, one entry per row) -> the bitmap b2ip_search_filtered reads: bit r & 31
    of 32-bit word r >> 5 is set when row r may be returned.  This is np.packbits(mask,
    bitorder="little") padded to whole words.  numpy in -> uint32 numpy array; torch tensor in ->
    int32 tensor (the same bits) on the tensor's device."""
    if _is_torch(allowed):
        import torch
        if allowed.dtype != torch.bool or allowed.dim() != 1:
            raise ValueError("allowed must be a 1-d bool tensor")
        n = allowed.shape[0]
        m = torch.zeros(-(-n // 32) * 32, dtype=torch.uint8, device=allowed.device)
        m[:n] = allowed
        shifts = torch.arange(8, dtype=torch.uint8, device=allowed.device)
        return (m.view(-1, 8) << shifts).sum(1, dtype=torch.uint8).view(torch.int32)
    a = np.asarray(allowed)
    if a.dtype != np.bool_ or a.ndim != 1:
        raise ValueError("allowed must be a 1-d bool array")
    b = np.packbits(a, bitorder="little")
    return np.pad(b, (0, -len(b) % 4)).view("<u4")


class Engine:
    def __init__(self, d: int, device: int = 0, store: str = "f32", shadow: Optional[str] = None):
        """store="f32": fp32 master rows (faiss semantics) + a 16-bit shadow for the coarse pass
        (`shadow` = "bf16" | "f16", default: the library's).  store="bf16" / "f16": the index keeps
        rows in that 16-bit type only (rounded at ingest unless handed in as such) and is exact
        w.r.t. those values with an fp32 rescore.  "bf16" is BASELINE config 4 (half the HBM);
        "f16" is lossless for the reference's default float16 embedding shards
        (generate_passage_embeddings.py:75-76), which src/index.py:27 merely widens."""
        self._lib = _lib.load()
        self._h = ctypes.c_void_p()
        self.store = store
        st = {"f32": STORE_F32, "bf16": STORE_BF16, "f16": STORE_F16}[store]
        check(self._lib.b2ip_create_ex(int(d), int(device), st, ctypes.byref(self._h)), None)
        self.d = int(d)
        self.device = int(device)
        if shadow is not None:
            if store != "f32":
                raise ValueError("shadow= applies to store='f32' only")
            self.set_option("shadow_f16", {"bf16": 0, "f16": 1}[shadow])

    # -- lifetime ------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.b2ip_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- configuration -------------------------------------------------------------
    def set_stream(self, cuda_stream: Optional[int]) -> None:
        """Run on this cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream)."""
        self._torch_stream = None
        check(self._lib.b2ip_set_stream(self._h, ctypes.c_void_p(cuda_stream or 0)), self._h)

    def use_torch_stream(self) -> None:
        import torch
        ptr = torch.cuda.current_stream(self.device).cuda_stream
        self.set_stream(ptr)
        self._torch_stream = ptr

    def _order_after_torch(self) -> None:
        """Work the caller queued on torch's current stream must be visible to the engine: nothing
        to do when the engine runs ON that stream (use_torch_stream), else wait for it."""
        import torch
        cur = torch.cuda.current_stream(self.device)
        if getattr(self, "_torch_stream", None) != cur.cuda_stream:
            cur.synchronize()

    def set_option(self, name: str, value: int) -> None:
        check(self._lib.b2ip_set_option(self._h, name.encode(), int(value)), self._h)

    def reserve(self, n_rows: int) -> None:
        check(self._lib.b2ip_reserve(self._h, int(n_rows)), self._h)

    def set_row_offset(self, offset: int) -> None:
        check(self._lib.b2ip_set_row_offset(self._h, int(offset)), self._h)

    def set_row_segments(self, segments) -> None:
        """segments: [(local_start, global_start, n), ...] in increasing order; the engine then
        reports GLOBAL row ids itself (one segment: a plain offset)."""
        if len(segments) <= 1:
            check(self._lib.b2ip_set_row_segments(self._h, 0, None, None), self._h)
            self.set_row_offset(segments[0][1] - segments[0][0] if segments else 0)
            return
        ls = np.ascontiguousarray([s[0] for s in segments], dtype=np.int64)
        gs = np.ascontiguousarray([s[1] for s in segments], dtype=np.int64)
        check(self._lib.b2ip_set_row_segments(self._h, len(segments), ctypes.c_void_p(ls.ctypes.data),
                                              ctypes.c_void_p(gs.ctypes.data)), self._h)

    @property
    def ntotal(self) -> int:
        return int(self._lib.b2ip_ntotal(self._h))

    # -- data ----------------------------------------------------------------------
    def add(self, rows) -> None:
        """Append rows [n,d]; float16 is widened exactly, anything else goes through float32
        (reference: `embeddings.astype('float32')`, src/index.py:27)."""
        if _is_torch(rows):
            import torch
            assert rows.is_cuda and rows.device.index == self.device, "tensor must live on the engine's GPU"
            ok = (torch.float16, torch.float32) + ((torch.bfloat16,) if self.store == "bf16" else ())
            if rows.dtype not in ok:
                rows = rows.float()
            rows = rows.contiguous()
            assert rows.dim() == 2 and rows.shape[1] == self.d, tuple(rows.shape)
            torch.cuda.current_stream(self.device).synchronize()
            dt = {torch.float16: B2IP_F16, torch.float32: B2IP_F32, torch.bfloat16: B2IP_BF16}[rows.dtype]
            check(self._lib.b2ip_add(self._h, rows.shape[0], ctypes.c_void_p(rows.data_ptr()), dt,
                                     MEM_DEVICE), self._h)
            return
        rows = np.asarray(rows)
        if rows.dtype not in (np.float16, np.float32):
            rows = rows.astype(np.float32)
        rows = np.ascontiguousarray(rows)
        if rows.ndim != 2 or rows.shape[1] != self.d:
            raise ValueError(f"expected [n,{self.d}] rows, got {rows.shape}")
        dt = B2IP_F16 if rows.dtype == np.float16 else B2IP_F32
        check(self._lib.b2ip_add(self._h, rows.shape[0], ctypes.c_void_p(rows.ctypes.data), dt,
                                 MEM_HOST), self._h)

    def export_rows(self, row0: int, n: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        if out is None:
            out = np.empty((n, self.d), dtype=np.float32)
        assert out.dtype == np.float32 and out.shape == (n, self.d) and out.flags["C_CONTIGUOUS"]
        check(self._lib.b2ip_export_rows(self._h, int(row0), int(n), ctypes.c_void_p(out.ctypes.data),
                                         MEM_HOST), self._h)
        return out

    # -- search --------------------------------------------------------------------
    def _search_call(self, nq, q_ptr, q_dtype, k, d_ptr, i_ptr, m, mem, allowed):
        if allowed is None:
            return self._lib.b2ip_search_ex(self._h, nq, q_ptr, q_dtype, k, d_ptr, i_ptr, m, mem)
        if len(allowed) != self.ntotal:
            raise ValueError(f"allowed has {len(allowed)} entries, the index holds {self.ntotal} rows")
        if _is_torch(allowed) and allowed.is_cuda and allowed.device.index != self.device:
            raise ValueError(f"allowed lives on {allowed.device}, the engine on cuda:{self.device}")
        bits = pack_allowed(allowed)
        # the bitmap crosses the ABI where the queries do (`mem`): wherever the mask was packed
        # (host numpy, a CPU or a CUDA tensor), move it there
        if mem == MEM_DEVICE:
            import torch
            if not _is_torch(bits):
                bits = torch.from_numpy(bits.view(np.int32))
            bits = bits.to(torch.device("cuda", self.device))
            self._order_after_torch()          # packed / copied on torch's stream
            ptr = bits.data_ptr()
        else:
            if _is_torch(bits):
                bits = bits.cpu().numpy()
            ptr = bits.ctypes.data
        return self._lib.b2ip_search_filtered(self._h, nq, q_ptr, q_dtype, k, ctypes.c_void_p(ptr), len(allowed),
                                              d_ptr, i_ptr, m, mem)

    def search(self, queries, k: int, mode: str = "auto", out=None, allowed=None) -> Tuple[object, object]:
        """(scores [nq,k] float32 descending, rows [nq,k] int64).  numpy in -> numpy out (host
        buffers cross the ABI, H2D/D2H inside the call); torch CUDA tensor in -> tensors out.
        `allowed` (bool, one entry per row: numpy, or a torch bool tensor on the engine's GPU)
        restricts the search to the rows it marks (faiss SearchParameters(sel=IDSelectorBitmap)):
        the answer is that of an index holding only those rows, with the original row ids; the
        tail is (-FLT_MAX, -1) when fewer than k allowed rows have a score."""
        m = _MODES[mode]
        k = int(k)
        if _is_torch(queries):
            import torch
            assert queries.is_cuda and queries.device.index == self.device
            # float16 queries cross the ABI as they are and are widened by the library (exact)
            q = queries.contiguous() if queries.dtype in (torch.float16, torch.float32) \
                else queries.float().contiguous()
            assert q.dim() == 2 and q.shape[1] == self.d, tuple(q.shape)
            nq = q.shape[0]
            if out is None:
                D = torch.empty((nq, k), dtype=torch.float32, device=q.device)
                I = torch.empty((nq, k), dtype=torch.int64, device=q.device)
            else:
                D, I = out
            self._order_after_torch()
            check(self._search_call(nq, ctypes.c_void_p(q.data_ptr()),
                                    B2IP_F16 if q.dtype == torch.float16 else B2IP_F32, k,
                                    ctypes.c_void_p(D.data_ptr()), ctypes.c_void_p(I.data_ptr()),
                                    m, MEM_DEVICE, allowed), self._h)
            return D, I
        q = np.asarray(queries)
        if q.dtype not in (np.float16, np.float32):
            q = q.astype(np.float32)
        q = np.ascontiguousarray(q)
        if q.ndim != 2 or q.shape[1] != self.d:
            raise ValueError(f"expected [nq,{self.d}] queries, got {q.shape}")
        nq = q.shape[0]
        if out is None:
            D = np.empty((nq, k), dtype=np.float32)
            I = np.empty((nq, k), dtype=np.int64)
        else:
            D, I = out
        check(self._search_call(nq, ctypes.c_void_p(q.ctypes.data),
                                B2IP_F16 if q.dtype == np.float16 else B2IP_F32, k,
                                ctypes.c_void_p(D.ctypes.data), ctypes.c_void_p(I.ctypes.data),
                                m, MEM_HOST, allowed), self._h)
        return D, I

    def range_search(self, queries, radius: float, mode: str = "auto"):
        """faiss `IndexFlatIP.range_search`: (lims [nq+1] int64, D [total] float32, I [total] int64);
        query i's hits are D/I[lims[i]:lims[i+1]], every row scoring strictly above `radius`, in
        ascending row order.  numpy in -> numpy out; torch CUDA tensor in -> CUDA tensors out."""
        m = _MODES[mode]
        if _is_torch(queries):
            import torch
            assert queries.is_cuda and queries.device.index == self.device
            q = queries.contiguous() if queries.dtype in (torch.float16, torch.float32) \
                else queries.float().contiguous()
            assert q.dim() == 2 and q.shape[1] == self.d, tuple(q.shape)
            lims = np.empty(q.shape[0] + 1, dtype=np.int64)
            self._order_after_torch()
            check(self._lib.b2ip_range_search(self._h, q.shape[0], ctypes.c_void_p(q.data_ptr()),
                                              B2IP_F16 if q.dtype == torch.float16 else B2IP_F32, float(radius), m,
                                              MEM_DEVICE, ctypes.c_void_p(lims.ctypes.data)), self._h)
            total = int(lims[-1])
            D = torch.empty(total, dtype=torch.float32, device=q.device)
            I = torch.empty(total, dtype=torch.int64, device=q.device)
            check(self._lib.b2ip_range_fetch(self._h, ctypes.c_void_p(D.data_ptr()), ctypes.c_void_p(I.data_ptr()),
                                             MEM_DEVICE), self._h)
            return torch.from_numpy(lims).to(q.device), D, I
        q = np.asarray(queries)
        if q.dtype not in (np.float16, np.float32):
            q = q.astype(np.float32)
        q = np.ascontiguousarray(q)
        if q.ndim != 2 or q.shape[1] != self.d:
            raise ValueError(f"expected [nq,{self.d}] queries, got {q.shape}")
        lims = np.empty(q.shape[0] + 1, dtype=np.int64)
        check(self._lib.b2ip_range_search(self._h, q.shape[0], ctypes.c_void_p(q.ctypes.data),
                                          B2IP_F16 if q.dtype == np.float16 else B2IP_F32, float(radius), m,
                                          MEM_HOST, ctypes.c_void_p(lims.ctypes.data)), self._h)
        total = int(lims[-1])
        D = np.empty(total, dtype=np.float32)
        I = np.empty(total, dtype=np.int64)
        check(self._lib.b2ip_range_fetch(self._h, ctypes.c_void_p(D.ctypes.data), ctypes.c_void_p(I.ctypes.data),
                                         MEM_HOST), self._h)
        return lims, D, I

    def enable_peer_access(self, peer_device: int) -> None:
        """Kernels of this engine's GPU may store into memory of `peer_device` (same process)."""
        check(self._lib.b2ip_enable_peer_access(self._h, int(peer_device)), self._h)

    def search_exchange(self, queries, k: int, ex, seq: int):
        """Local search + peer-direct exchange + merge in one call (b2ip_search_exchange).
        `ex`: _lib.Exchange of this parity.  Returns (D, I, status): the GLOBAL top-k on this
        rank's device -- of every query (ex.gather_mode == GATHER_ALL) or of the queries this
        rank owns, `shard_bounds(nq, world, rank)`, compactly (GATHER_OWNER) -- and the number of
        overflowed queries over all ranks (non-zero: repeat the search through the all-gather path)."""
        import torch
        q = queries.float().contiguous()
        assert q.is_cuda and q.device.index == self.device and q.dim() == 2 and q.shape[1] == self.d
        nq, k = q.shape[0], int(k)
        n_out = nq
        if ex.gather_mode == _lib.GATHER_OWNER:
            per = -(-nq // ex.world)
            lo = min(ex.rank * per, nq)
            n_out = min(lo + per, nq) - lo
        D = torch.empty((n_out, k), dtype=torch.float32, device=q.device)
        I = torch.empty((n_out, k), dtype=torch.int64, device=q.device)
        status = ctypes.c_int64(0)
        self._order_after_torch()
        check(self._lib.b2ip_search_exchange(self._h, nq, ctypes.c_void_p(q.data_ptr()), k, ctypes.byref(ex),
                                             ctypes.c_uint32(seq & 0xFFFFFFFF), ctypes.c_void_p(D.data_ptr()),
                                             ctypes.c_void_p(I.data_ptr()), ctypes.byref(status)), self._h)
        return D, I, int(status.value)

    def upload(self, dst, src: np.ndarray) -> None:
        """dst (torch CUDA tensor on this engine's device) <- src (host array of the same byte
        size), through the handle's pinned double-buffered staging."""
        src = np.ascontiguousarray(src)
        assert dst.is_cuda and dst.device.index == self.device and dst.is_contiguous()
        assert dst.numel() * dst.element_size() == src.nbytes
        check(self._lib.b2ip_copy_to_device(self._h, ctypes.c_void_p(dst.data_ptr()),
                                            ctypes.c_void_p(src.ctypes.data), src.nbytes), self._h)

    def download(self, src, dst: np.ndarray) -> None:
        """dst (C-contiguous host array) <- src (torch CUDA tensor on this engine's device)."""
        assert src.is_cuda and src.device.index == self.device and src.is_contiguous()
        assert dst.flags["C_CONTIGUOUS"] and src.numel() * src.element_size() == dst.nbytes
        import torch
        torch.cuda.current_stream(self.device).synchronize()
        check(self._lib.b2ip_copy_to_host(self._h, ctypes.c_void_p(dst.ctypes.data),
                                          ctypes.c_void_p(src.data_ptr()), dst.nbytes), self._h)

    def stats(self) -> dict:
        s = Stats()
        check(self._lib.b2ip_stats(self._h, ctypes.byref(s)), self._h)
        return s.as_dict()

    def debug_coarse_scores(self, queries, row0: int, n_rows: int):
        """Test hook: raw tcgen05 bf16 scores [nq,n_rows] (torch CUDA tensors only)."""
        import torch
        q = queries.float().contiguous()
        out = torch.empty((q.shape[0], n_rows), dtype=torch.float32, device=q.device)
        torch.cuda.current_stream(self.device).synchronize()
        check(self._lib.b2ip_debug_coarse_scores(self._h, q.shape[0], ctypes.c_void_p(q.data_ptr()),
                                                 int(row0), int(n_rows), ctypes.c_void_p(out.data_ptr())),
              self._h)
        return out


def merge_topk(scores, rows, k: int):
    """Device merge of per-shard results: scores/rows torch CUDA tensors [G,nq,k] -> ([nq,k],[nq,k]).
    The G lists may be strided views (e.g. slices of one packed all-gather buffer) as long as
    each [nq,k] list is itself contiguous."""
    import torch
    lib = _lib.load()
    G, nq, kk = scores.shape
    assert kk == k and rows.shape == scores.shape
    if not scores[0].is_contiguous() or (G > 1 and scores.stride(0) < nq * k):
        scores = scores.contiguous()
    if not rows[0].is_contiguous() or (G > 1 and rows.stride(0) < nq * k):
        rows = rows.contiguous()
    D = torch.empty((nq, k), dtype=torch.float32, device=scores.device)
    I = torch.empty((nq, k), dtype=torch.int64, device=scores.device)
    stream = torch.cuda.current_stream(scores.device)
    check(lib.b2ip_merge_topk_strided(
        scores.device.index, ctypes.c_void_p(stream.cuda_stream), nq, k, G,
        ctypes.c_void_p(scores.data_ptr()), ctypes.c_void_p(rows.data_ptr()),
        scores.stride(0) if G > 1 else nq * k, rows.stride(0) if G > 1 else nq * k,
        ctypes.c_void_p(D.data_ptr()), ctypes.c_void_p(I.data_ptr())), None)
    return D, I
