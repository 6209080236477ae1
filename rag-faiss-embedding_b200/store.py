"""FAISSVectorStore -- host-side mirror of the reference's vector-store wrapper (faiss_store.py:10-128)
on top of the B200 index: same constructor arguments, attributes (dimension, index_path, doc_ids,
index), method names, argument meaning, return shapes and error behaviour, so database.py:31,85,94,
query.py:36 and initialize_rag.py:57-61 work against it as they do against the original.

Differences, all additive: `search_many` (a batch of queries in one device call -- the reference
forces nq=1 at faiss_store.py:61), `remove_documents`, `metric="ip"`, and the instance is not forced to be a process-wide
singleton unless `singleton=True` is requested through `get_instance()`.
"""
from __future__ import annotations

import logging
import os
import pickle
from typing import List, Optional, Sequence, Tuple

import numpy as np

from .index import IDSelectorBatch, IndexFlatIP, IndexFlatL2, SearchParameters, read_index, write_index

log = logging.getLogger("b200flat.store")


class FAISSVectorStore:
    _shared: Optional["FAISSVectorStore"] = None

    def __init__(self, dimension: int = 384, index_path: str = "data/faiss_index.bin", metric: str = "l2",
                 device: Optional[int] = None):
        self.dimension = dimension
        self.index_path = index_path
        self.metric = metric.lower()
        self._device = device
        self.doc_ids: List[int] = []
        self.index = self._new_index()
        if os.path.exists(index_path):
            self.load_index()
        log.info("vector store ready: d=%d, %d vectors", dimension, self.index.ntotal)

    @classmethod
    def get_instance(cls, *args, **kwargs) -> "FAISSVectorStore":
        """Process-wide instance, the reference's singleton behaviour (faiss_store.py:14-17,21-22)."""
        if cls._shared is None:
            cls._shared = cls(*args, **kwargs)
        return cls._shared

    def _new_index(self):
        kind = IndexFlatIP if self.metric in ("ip", "inner_product") else IndexFlatL2
        return kind(self.dimension, device=self._device)

    # faiss_store.py:36-47
    def add_vectors(self, vectors, ids: Sequence[int]):
        arr = np.asarray(vectors, dtype=np.float32)
        if arr.ndim == 1:
            arr = arr[None, :]
        self.doc_ids.extend(ids)
        self.index.add(arr)
        log.info("added %d vectors", len(ids))

    def _doc_params(self, doc_ids) -> dict:
        """search() keywords restricting a search to the rows of the documents doc_ids (None: every row)."""
        if doc_ids is None:
            return {}
        want = set(doc_ids)
        rows = np.asarray([i for i, d in enumerate(self.doc_ids) if d in want], dtype=np.int64)
        return {"params": SearchParameters(sel=IDSelectorBatch(rows))}

    # faiss_store.py:49-81 -- nq is forced to 1, padding rows are dropped, every failure is swallowed.
    # doc_ids (keyword only, no reference counterpart): search only the rows of those documents.
    def search(self, query_vector, k: int = 5, *, doc_ids: Optional[Sequence[int]] = None) -> Tuple[np.ndarray, List[int]]:
        try:
            q = np.asarray(query_vector, dtype=np.float32).reshape(1, -1)
            dist, rows = self.index.search(q, k, **self._doc_params(doc_ids))
            kept_d, kept_ids = [], []
            for pos, row in enumerate(rows[0]):
                if row != -1 and row < len(self.doc_ids):
                    kept_ids.append(self.doc_ids[row])
                    kept_d.append(dist[0][pos])
            return np.array(kept_d), kept_ids
        except Exception as exc:  # noqa: BLE001 - the reference returns empty results on any error
            log.error("search failed: %s", exc)
            return np.array([]), []

    def search_many(self, query_vectors, k: int = 5, *, doc_ids: Optional[Sequence[int]] = None
                    ) -> Tuple[np.ndarray, List[List[int]]]:
        """Batched variant (SURVEY 8f rank 3): [nq, d] queries -> (D [nq, k], doc ids per query).  doc_ids: search
        only the rows of those documents."""
        q = np.asarray(query_vectors, dtype=np.float32)
        if q.ndim == 1:
            q = q[None, :]
        dist, rows = self.index.search(q, k, **self._doc_params(doc_ids))
        mapped = [[self.doc_ids[r] for r in row if r != -1 and r < len(self.doc_ids)] for row in rows]
        return dist, mapped

    def remove_documents(self, doc_ids: Sequence[int]) -> int:
        """Removes every row whose document id is in doc_ids, and the same positions from self.doc_ids, so that rows and
        ids stay aligned (and save_index writes a .mapping that matches the file).  Returns the number of rows removed."""
        drop = set(doc_ids)
        rows = [i for i, d in enumerate(self.doc_ids) if d in drop]
        if not rows:
            return 0
        n = self.index.remove_ids(np.asarray(rows, dtype=np.int64))
        gone = set(rows)
        self.doc_ids = [d for i, d in enumerate(self.doc_ids) if i not in gone]
        log.info("removed %d vectors", n)
        return n

    # faiss_store.py:83-97
    def save_index(self, filepath: Optional[str] = None):
        path = filepath or self.index_path
        folder = os.path.dirname(path)
        if folder:
            os.makedirs(folder, exist_ok=True)
        write_index(self.index, path)
        with open(path + ".mapping", "wb") as fh:
            pickle.dump(self.doc_ids, fh)
        log.info("saved index + mapping to %s", path)

    # faiss_store.py:99-122 -- a missing mapping means sequential ids; errors propagate
    def load_index(self, filepath: Optional[str] = None):
        path = filepath or self.index_path
        self.index = read_index(path, device=self._device)
        mapping = path + ".mapping"
        if os.path.exists(mapping):
            with open(mapping, "rb") as fh:
                self.doc_ids = pickle.load(fh)
        else:
            self.doc_ids = list(range(self.index.ntotal))
            log.warning("no mapping file next to %s; using sequential ids", path)

    # faiss_store.py:124-128
    def reset(self):
        self.index = self._new_index()
        self.doc_ids = []
