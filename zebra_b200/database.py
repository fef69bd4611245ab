"""Database: the host mirror of /root/reference/src/database/core.rs:55-381 for the three index call sites
(insert_records :245-254, remove :205-213, query_vectors :290-313).

The document store of the reference (lz4 files, core.rs:322-380) is host I/O outside the hot path; documents are kept
in an in-memory map here so the API round-trips.  `save_database` / `open` write and read the reference's `.zebra` file
(core.rs:92-104, :183-190) next to a dump of the index's two key-value partitions (interchange.py).
"""
from __future__ import annotations

import uuid as _uuid
from typing import Dict, List, Optional, Sequence

import numpy as np

from .distance import CosineDistance, _DeviceMetric
from .index import LSHIndex, LSHIndexOptions, _bytes_to_ids


class DatabaseEmbeddingModel:
    """model/core.rs:12-37: `embed_documents(&self, documents) -> Vec<Embedding<N>>`.  Out of scope; kept so
    Database stays generic over a model."""

    def embed_documents(self, documents: Sequence[bytes]) -> np.ndarray:  # pragma: no cover - interface
        raise NotImplementedError("no embedding model on the device path (BASELINE configs use raw vectors)")


class Database:
    """core.rs:55-64.  `index` is public like the reference's `pub index: LSHIndex<N>` (core.rs:62)."""

    def __init__(self, dim: int, metric: Optional[_DeviceMetric] = None, model: Optional[DatabaseEmbeddingModel] = None,
                 index_options: Optional[LSHIndexOptions] = None, device: int = 0, seed: int = 0):
        self.dim = dim
        self.metric = metric or CosineDistance()
        self.model = model or DatabaseEmbeddingModel()
        self.index_options = index_options or LSHIndexOptions()
        self.uuid = _uuid.uuid4()
        self.index = LSHIndex(dim, self.index_options, self.metric, device=device, seed=seed)
        self._documents: Dict[_uuid.UUID, bytes] = {}
        self.path = ""

    @classmethod
    def new(cls, dim: int, index_options: LSHIndexOptions, **kw) -> "Database":  # core.rs:110
        return cls(dim, index_options=index_options, **kw)

    def default_database_path(self) -> str:  # core.rs:80-82
        return f"{self.uuid.hex}.zebra"

    def save_database(self, path: Optional[str] = None) -> None:  # core.rs:183-190
        """Writes `path` = bincode(legacy) of DatabaseInner, byte for byte what the reference writes, and
        `path + ".store"` = the index's `trees` and `embeddings` partitions (values as the reference stores them)."""
        from . import interchange

        path = path or self.path or self.default_database_path()
        zebra = interchange.zebra_file_encode(self.uuid, self.metric, self.index_options.max_node_size,
                                              self.index_options.num_trees)
        with open(path, "wb") as f:
            f.write(zebra)
        self.index.save_store(path + ".store", zebra)
        self.path = path

    @classmethod
    def open(cls, path: str, dim: int, metric: Optional[_DeviceMetric] = None, **kw) -> "Database":  # core.rs:92-104
        """`dim` and `metric` are the reference's type parameters N and Met (the file does not carry them)."""
        from . import interchange

        metric = metric or CosineDistance()
        with open(path, "rb") as f:
            db_uuid, power, mns, nt = interchange.zebra_file_decode(f.read(), metric)
        if hasattr(metric, "power"):
            metric.power = power
        db = cls(dim, metric, index_options=LSHIndexOptions(mns, nt), **kw)
        db.uuid, db.path = db_uuid, path
        db.index.load_store(path + ".store")
        return db

    def clear_database(self) -> None:  # core.rs:194-198
        self.index.clear()
        self._documents.clear()

    def remove(self, embedding_ids: Sequence[_uuid.UUID]) -> None:  # core.rs:205-213
        removed = self.index.remove(embedding_ids)
        for i in removed:
            self._documents.pop(i, None)

    def deduplicate(self) -> None:  # core.rs:216-224
        for i in self.index.deduplicate():
            self._documents.pop(i, None)

    def insert_documents(self, documents: Sequence[bytes]) -> None:  # core.rs:232-235
        self.insert_records(self.model.embed_documents(documents), documents)

    def insert_records(self, embeddings, documents: Sequence[bytes]) -> List[_uuid.UUID]:  # core.rs:245-254
        embeddings = np.ascontiguousarray(embeddings, dtype=np.float32).reshape(-1, self.dim)
        if len(documents) != embeddings.shape[0]:
            raise ValueError("one document per embedding")
        ids = self.index.add(embeddings)
        for i, d in zip(ids, documents):
            self._documents[i] = bytes(d)
        return ids  # the reference discards them (survey Q9); returned here for convenience

    def query_documents(self, documents: Sequence[bytes], number_of_results: int):  # core.rs:267-277
        if self.index.no_vectors():
            return {}
        return self.query_vectors(self.model.embed_documents(documents), number_of_results)

    def query_vectors(self, vectors, number_of_results: int, probes: int = 0) -> Dict[int, Dict[_uuid.UUID, bytes]]:  # core.rs:290-313
        """probes > 0: multi-probe search (LSHIndex.search_batch); 0 is the reference's query."""
        if self.index.no_vectors():
            return {}
        vectors = np.ascontiguousarray(vectors, dtype=np.float32).reshape(-1, self.dim)
        ids, _, _, counts = self.index.search_batch(vectors, number_of_results, probes=probes)  # ONE batched device call
        out: Dict[int, Dict[_uuid.UUID, bytes]] = {}
        for q in range(vectors.shape[0]):
            out[q] = {i: self._documents.get(i, b"") for i in _bytes_to_ids(ids[q, : int(counts[q])])}
        return out
