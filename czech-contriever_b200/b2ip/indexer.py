"""Drop-in replacement for the reference's `src/index.py` (Indexer over faiss.IndexFlatIP).

Same class, methods, prints and return types as reference src/index.py:15-73 (re-exported under
the reference's module path by `czech-contriever_b200/src/index.py`, and installed over the
reference's own `src.index` by `python -m b2ip.dropin <script>`);
the faiss object is replaced by `b2ip.Engine` (libb2ip.so, B200 only).  Differences, all
deliberate:
  * `n_subquantizers > 0` (faiss.IndexPQ, src/index.py:18-19) raises: approximate search is
    not on this path and there is no CPU fallback.
  * `index_batch_size` is a hint: queries are independent, the engine batches them itself.
  * the id mapping of src/index.py:44 (nq*k Python str() calls) runs in C (csrc/hostmap.c),
    pipelined behind the GPU search chunk by chunk -- same strings, same `[-1]` = last-id
    quirk for the -1 padding the reference has when the index holds fewer than k rows.
  * `search_knn` also takes a torch CUDA tensor (the query encoder's output, left on the GPU).
  * storage (`store=` / env B2IP_STORE, default "auto"): the reference widens whatever it is
    given to float32 (src/index.py:27).  Its default pipeline hands in float16 shards
    (generate_passage_embeddings.py:75-76); widening is exact, so "auto" keeps such rows as
    fp16 in HBM (a third of the memory, identical results) and moves the whole index to fp32
    master rows the first time a chunk arrives that is not float16.
  * devices (`device=` / env B2IP_DEVICES): an int is one GPU (default: B2IP_DEVICE, else
    LOCAL_RANK, else 0); "all" or a list row-shards the index over those GPUs from this single
    process (`b2ip.multi.MultiGpuEngine`) -- the reference driver is single-process, so this
    is how an unmodified passage_retrieval.py uses a whole 8-GPU box.
"""
import os
import pickle
from typing import List, Tuple

import numpy as np

from ._lib import load_hostmap
from .engine import Engine, _is_torch
from .ingest import prefetch
from .multi import MultiGpuEngine
from .faiss_io import stream_flat_ip_rows, write_flat_ip


class Indexer(object):

    def __init__(self, vector_sz, n_subquantizers=0, n_bits=8, device=None, store=None):
        if n_subquantizers > 0:
            raise NotImplementedError(
                "IndexPQ (n_subquantizers > 0) is approximate search; the B200 engine implements "
                "exact IndexFlatIP only and has no CPU fallback")
        if device is None and os.environ.get("B2IP_DEVICES"):
            device = os.environ["B2IP_DEVICES"]
        if isinstance(device, str) and device != "all":
            device = [int(x) for x in device.split(",") if x.strip() != ""]
        if device is None:
            device = int(os.environ.get("B2IP_DEVICE", os.environ.get("LOCAL_RANK", "0")))
        if store is None:
            store = os.environ.get("B2IP_STORE", "auto")
        if store not in ("auto", "f32", "f16"):
            raise ValueError("store must be 'auto', 'f32' or 'f16' (an explicit 'f16' rounds fp32 rows)")
        self.vector_sz = vector_sz
        self.device = device
        self.store = store
        self.index = self._new_engine(vector_sz, "f16" if store == "f16" else "f32")
        self.index_id_to_db_id = []
        self.knn_chunk = 32768        # queries per pipelined search_knn chunk (env B2IP_KNN_CHUNK)
        self._id_rows = None          # str(db_id) -> rows, built by the first filtered search_knn

    @classmethod
    def from_engine(cls, engine, ids=None, store=None) -> "Indexer":
        """The drop-in object around an engine that already holds the rows (e.g. one built
        from device tensors): `ids` become `index_id_to_db_id`."""
        self = cls.__new__(cls)
        self.vector_sz, self.store = engine.d, store or engine.store
        self.device = getattr(engine, "devices", None) or engine.device
        self.index = engine
        self.index_id_to_db_id = list(ids) if ids is not None else []
        self.knn_chunk = 32768
        self._id_rows = None
        return self

    def _new_engine(self, d, store):
        if self.device == "all":
            return MultiGpuEngine(d, None, store=store)
        if isinstance(self.device, (list, tuple)):
            return MultiGpuEngine(d, self.device, store=store) if len(self.device) > 1 \
                else Engine(d, self.device[0], store=store)
        return Engine(d, self.device, store=store)

    def _is_f16(self, embeddings):
        dt = getattr(embeddings, "dtype", None)
        return dt is not None and str(dt).endswith("float16") and not str(dt).endswith("bfloat16")

    def _restore(self, store):
        """Moves the rows held so far into an engine with another storage type (exact:
        fp16 -> fp32 widening)."""
        new = self._new_engine(self.vector_sz, store)
        n = self.index.ntotal
        new.reserve(n)
        for r0 in range(0, n, 1 << 18):
            new.add(self.index.export_rows(r0, min(1 << 18, n - r0)))
        self.index.close()
        self.index = new

    def index_data(self, ids, embeddings):
        self._update_id_mapping(ids)
        self._id_rows = None
        # reference: embeddings.astype('float32'); fp16 is widened on the GPU (exact)
        if self.store == "auto":
            if self._is_f16(embeddings):
                if self.index.ntotal == 0 and self.index.store != "f16":
                    self.index.close()
                    self.index = self._new_engine(self.vector_sz, "f16")
            elif self.index.store == "f16":
                self._restore("f32")
        self.index.add(embeddings)

        print(f'Total data indexed {len(self.index_id_to_db_id)}')

    def allowed_mask(self, allowed_ids) -> np.ndarray:
        """Bool mask over the indexed rows: True for every row whose external id, as `str`, is in
        `allowed_ids` (duplicated ids: all their rows).  Unknown ids are ignored, as a faiss
        selector ignores ids the index does not hold.  The id -> rows lookup is built on the first
        call and kept until `index_data` or `deserialize_from` changes the ids."""
        if self._id_rows is None:
            first, dups = {}, {}
            for r, s in enumerate(map(str, self.index_id_to_db_id)):
                j = first.setdefault(s, r)
                if j != r:
                    dups.setdefault(s, [j]).append(r)
            self._id_rows = (first, dups)
        first, dups = self._id_rows
        mask = np.zeros(len(self.index_id_to_db_id), dtype=bool)
        rows = []
        for a in set(map(str, allowed_ids)):
            if a in dups:
                rows.extend(dups[a])
            elif a in first:
                rows.append(first[a])
        mask[np.asarray(rows, dtype=np.int64)] = True
        return mask

    def search_knn(self, query_vectors: np.array, top_docs: int, index_batch_size: int = 2048,
                   allowed_ids=None) -> List[Tuple[List[object], List[float]]]:
        """reference src/index.py:34-46, same return value: nq tuples (list of k external ids as
        `str`, float32 score row), rows score-descending.  `query_vectors` may be a numpy array
        (float16 / float32 are handed to the library as they are -- float16 is widened on the
        GPU, which is what `astype('float32')` computes -- anything else goes through float32)
        or a torch tensor; a CUDA tensor is searched where it lies (no host round trip of the
        queries: SURVEY 8f N4, the encoder's output can stay on the device).

        The queries are searched in chunks on a background thread while this thread maps the
        previous chunk's rows to external ids (csrc/hostmap.c: the reference's nq*k str() loop
        in C), so the host half of the call hides behind the GPU half.

        `allowed_ids` (an iterable of external ids, matched as `str`) restricts the search to
        those passages (faiss SearchParameters(sel=...)); each tuple then holds only the real
        results, fewer than `top_docs` when fewer passages are allowed, with no padding."""
        q = query_vectors
        on_device = False
        if _is_torch(q):
            q = q.detach()
            if q.is_cuda:
                on_device = True
            else:
                q = q.numpy()
        if not on_device:
            q = np.asarray(q)
            if q.dtype not in (np.float16, np.float32):
                q = q.astype('float32')
        nq = len(q)
        if nq == 0:
            return []
        ids = self.index_id_to_db_id
        if not isinstance(ids, list):
            ids = list(ids)
        map_ids = load_hostmap().map_ids
        chunk = max(1, int(os.environ.get("B2IP_KNN_CHUNK", self.knn_chunk)))
        index = self.index
        allowed = None if allowed_ids is None else self.allowed_mask(allowed_ids)
        if allowed is not None and not ids:
            return [([], np.empty(0, np.float32)) for _ in range(nq)]

        def searches():
            for s in range(0, nq, chunk):
                D, I = index.search(q[s:s + chunk], top_docs) if allowed is None else \
                    index.search(q[s:s + chunk], top_docs, allowed=allowed)
                if on_device:
                    Dn = np.empty(tuple(D.shape), np.float32)
                    In = np.empty(tuple(I.shape), np.int64)
                    index.download(D.contiguous(), Dn)
                    index.download(I.contiguous(), In)
                    D, I = Dn, In
                yield D, I

        result = []
        # convert to external ids (negative rows index from the end, like the reference's
        # `index_id_to_db_id[-1]` for faiss's -1 padding; an empty id list raises IndexError)
        for scores, indexes in prefetch(searches(), depth=2):
            part = map_ids(ids, indexes, indexes.shape[0], indexes.shape[1], list(scores))
            if allowed is not None:
                # the -1 padding sits at the tail of a row: keep the real results only
                n_real = (indexes >= 0).sum(axis=1).tolist()
                part = [(i[:c], s[:c]) for (i, s), c in zip(part, n_real)]
            result.extend(part)
        return result

    def search_range(self, query_vectors, radius: float) -> List[Tuple[List[object], np.ndarray]]:
        """Every indexed passage whose inner product with the query is strictly above `radius`
        (faiss `IndexFlatIP.range_search`).  Takes what `search_knn` takes and returns one tuple
        per query, like `search_knn`: (external ids as `str`, float32 scores), score-descending,
        equal scores in insertion order."""
        q = query_vectors
        if _is_torch(q):
            q = q.detach()
            if not q.is_cuda:
                q = q.numpy()
        if not _is_torch(q):
            q = np.asarray(q)
            if q.dtype not in (np.float16, np.float32):
                q = q.astype('float32')
        if len(q) == 0:
            return []
        lims, D, I = self.index.range_search(q, radius)
        if _is_torch(lims):
            lims, D, I = lims.cpu().numpy(), D.cpu().numpy(), I.cpu().numpy()
        ids = self.index_id_to_db_id
        qi = np.repeat(np.arange(len(lims) - 1), np.diff(lims))
        order = np.lexsort((I, -D.astype(np.float64), qi))
        D, I = D[order], I[order]
        return [([str(ids[r]) for r in I[lims[i]:lims[i + 1]].tolist()], D[lims[i]:lims[i + 1]])
                for i in range(len(lims) - 1)]

    def serialize(self, dir_path):
        index_file = os.path.join(dir_path, 'index.faiss')
        meta_file = os.path.join(dir_path, 'index_meta.faiss')
        print(f'Serializing index to {index_file}, meta data to {meta_file}')

        write_flat_ip(index_file, self.vector_sz, self.index.ntotal, self.index.export_rows)
        with open(meta_file, mode='wb') as f:
            pickle.dump(self.index_id_to_db_id, f)

    def deserialize_from(self, dir_path):
        index_file = os.path.join(dir_path, 'index.faiss')
        meta_file = os.path.join(dir_path, 'index_meta.faiss')
        print(f'Loading index from {index_file}, meta data from {meta_file}')

        d, ntotal, blocks = stream_flat_ip_rows(index_file)
        index = self._new_engine(d, "f16" if self.store == "f16" else "f32")
        index.reserve(ntotal)
        for block in blocks:
            index.add(block)
        self.index.close()
        self.index = index
        self.vector_sz = d
        print('Loaded index of type %s and size %d', type(self.index), self.index.ntotal)

        with open(meta_file, "rb") as reader:
            self.index_id_to_db_id = pickle.load(reader)
        self._id_rows = None
        assert len(
            self.index_id_to_db_id) == self.index.ntotal, 'Deserialized index_id_to_db_id should match faiss index size'

    def _update_id_mapping(self, db_ids: List):
        self.index_id_to_db_id.extend(db_ids)
