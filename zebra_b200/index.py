"""LSHIndex: the host mirror of /root/reference/src/database/index/lsh.rs:122-566 over the CUDA library.

Same method names, argument meaning and error behaviour as the reference type (errors raise instead of
returning ``anyhow::Result``).  All compute happens in libzebra_b200.so; this file only marshals buffers.
"""
from __future__ import annotations

import ctypes as C
import uuid as _uuid
import weakref
from dataclasses import dataclass
from typing import Iterable, List, Optional, Sequence, Set, Tuple

import numpy as np

from . import _ffi
from .distance import _DeviceMetric


@dataclass
class LSHIndexOptions:
    """lsh.rs:122-138 (defaults 5 / 15)."""
    max_node_size: int = 5
    num_trees: int = 15


class Forest:
    """Flat forest arrays exchanged through zb_index_export_forest / zb_index_load_forest."""

    def __init__(self, nodes, roots, coef, cst, leaf_off, members):
        self.nodes = np.ascontiguousarray(nodes, dtype=np.int32).reshape(-1, 4)
        self.roots = np.ascontiguousarray(roots, dtype=np.int32)
        self.coef = np.ascontiguousarray(coef, dtype=np.float32)
        self.cst = np.ascontiguousarray(cst, dtype=np.float32)
        self.leaf_off = np.ascontiguousarray(leaf_off, dtype=np.int64)
        self.members = np.ascontiguousarray(members, dtype=np.uint64)


def _ids_to_bytes(ids: Iterable) -> np.ndarray:
    out = bytearray()
    for i in ids:
        out += i.bytes if isinstance(i, _uuid.UUID) else bytes(i)
    return np.frombuffer(bytes(out), dtype=np.uint8).copy()


def _bytes_to_ids(raw: np.ndarray) -> List[_uuid.UUID]:
    b = raw.tobytes()
    return [_uuid.UUID(bytes=b[i:i + 16]) for i in range(0, len(b), 16)]


ROWSET_EXCLUDE = 1  # ZB_ROWSET_EXCLUDE


class RowSet:
    """A fixed set of rows of one LSHIndex, for restricted search (`within=` of every search form, DESIGN 3.10).

    Made by `LSHIndex.rowset`.  A restricted search returns exactly what the plain search would return if every live row
    outside the set had been removed, without changing the index for anyone else.  The set is fixed when it is made: rows
    added later are never in it; rows removed later are excluded at call time; inserts, leaf splits and deduplicate are
    taken into account.  After `clear`, `load_forest`, `load_flat` or `import_store` (which reuse ordinals) a search with it
    raises ZebraError (ZB_ERR_STATE).  It holds device memory: `close()` it, or use it as a context manager.  It keeps its
    index alive; closing the index closes its rowsets.

    `count`: ordinals in the set.  `found`: for a set made from ids, which ids the index knows (unknown ones are ignored)."""

    def __init__(self, index: "LSHIndex", handle: C.c_void_p, count: int, found: Optional[np.ndarray] = None):
        self.index = index
        self._h = handle
        self.count = count
        self.found = found

    def close(self) -> None:
        if getattr(self, "_h", None) and self._h.value:
            _ffi.check(_ffi.lib().zb_rowset_destroy(self._h))
            self._h = C.c_void_p()

    def __enter__(self) -> "RowSet":
        return self

    def __exit__(self, *exc) -> None:
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class LSHIndex:
    """lsh.rs:145-148.  `metric` fixes the distance the device index scores with (the reference passes the
    metric to search(); a device index is built for ONE metric of distance.rs -- the fused leaf-tile scan serves
    Cosine / L2Squared / L2, the ten scalar metrics go through the gather path)."""

    def __init__(self, dim: int, options: Optional[LSHIndexOptions] = None, metric: Optional[_DeviceMetric] = None,
                 device: int = 0, seed: int = 0, shard_rank: int = 0, shard_count: int = 1):
        from .distance import CosineDistance

        self.dim = int(dim)
        self.options = options or LSHIndexOptions()
        self.metric = metric or CosineDistance()
        if not isinstance(self.metric, _DeviceMetric):
            raise TypeError("metric must be one of the zebra_b200.distance metric objects")
        self.device = device
        self.metric.device = device
        o = _ffi.Options()
        o.dim, o.metric, o.metric_power = self.dim, self.metric.METRIC, self.metric.power
        o.max_node_size, o.num_trees = self.options.max_node_size, self.options.num_trees
        o.device, o.seed = device, seed
        o.shard_rank, o.shard_count = shard_rank, shard_count
        self._h = C.c_void_p()
        self._rowsets = weakref.WeakSet()
        _ffi.check(_ffi.lib().zb_index_create(C.byref(o), C.byref(self._h)))

    # lsh.rs:162
    @classmethod
    def new(cls, dim: int, options: LSHIndexOptions, **kw) -> "LSHIndex":
        return cls(dim, options, **kw)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            for rs in list(getattr(self, "_rowsets", ())):  # a rowset belongs to its index: it goes first
                rs.close()
            _ffi.lib().zb_index_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def save(self) -> None:
        """lsh.rs:170-172 (fjall `persist`): the key-value engine is the host's; `save_store` / `export_tree_blobs` /
        `export_rows` produce the values it would persist."""

    # ---------------------------------------------------------------- lsh.rs:440-466
    def add(self, embeddings, ids: Optional[Sequence] = None) -> List[_uuid.UUID]:
        return _bytes_to_ids(self.add_raw(embeddings, ids)[0])

    def add_raw(self, embeddings, ids: Optional[Sequence] = None) -> Tuple[np.ndarray, np.ndarray]:
        """Returns (ids as [n,16] uint8, ordinals as [n] uint64)."""
        rows = np.ascontiguousarray(embeddings, dtype=np.float32).reshape(-1, self.dim)
        n = rows.shape[0]
        out_ids = np.empty((n, 16), dtype=np.uint8)
        out_ord = np.empty(n, dtype=np.uint64)
        idb = _ids_to_bytes(ids) if ids is not None else None
        if idb is not None and idb.size != 16 * n:
            raise ValueError("ids must hold one 16-byte id per row")
        _ffi.check(_ffi.lib().zb_index_add(self._h, n, rows.ctypes.data, idb.ctypes.data if idb is not None else None,
                                           out_ids.ctypes.data, out_ord.ctypes.data))
        return out_ids, out_ord

    def add_device(self, d_rows_ptr: int, n: int) -> np.ndarray:
        """Rows already resident in HBM (n*dim f32 at d_rows_ptr).  Returns ordinals."""
        out_ord = np.empty(n, dtype=np.uint64)
        _ffi.check(_ffi.lib().zb_index_add_device(self._h, n, d_rows_ptr, None, None, out_ord.ctypes.data))
        return out_ord

    def add_owned_device(self, d_rows_ptr: int, ordinals, total_n: int) -> None:
        ordinals = np.ascontiguousarray(ordinals, dtype=np.uint64)
        _ffi.check(_ffi.lib().zb_index_add_owned_device(self._h, ordinals.size, d_rows_ptr, ordinals.ctypes.data, total_n))

    # ---------------------------------------------------------------- lsh.rs:473-503
    def remove(self, embedding_ids: Sequence) -> Set[_uuid.UUID]:
        ids = list(embedding_ids)
        idb = _ids_to_bytes(ids)
        flags = np.zeros(len(ids), dtype=np.uint8)
        _ffi.check(_ffi.lib().zb_index_remove(self._h, len(ids), idb.ctypes.data if len(ids) else None, flags.ctypes.data))
        return {i if isinstance(i, _uuid.UUID) else _uuid.UUID(bytes=bytes(i)) for i, f in zip(ids, flags) if f}

    def remove_ordinals(self, ordinals) -> np.ndarray:
        ordinals = np.ascontiguousarray(ordinals, dtype=np.uint64)
        flags = np.zeros(ordinals.size, dtype=np.uint8)
        _ffi.check(_ffi.lib().zb_index_remove_ordinals(self._h, ordinals.size, ordinals.ctypes.data, flags.ctypes.data))
        return flags.astype(bool)

    # ---------------------------------------------------------------- lsh.rs:270-288
    def deduplicate(self) -> Set[_uuid.UUID]:
        return set(_bytes_to_ids(self.deduplicate_raw()[0]))

    def deduplicate_raw(self) -> Tuple[np.ndarray, np.ndarray]:
        """Returns (ids as [n,16] uint8, ordinals as [n] uint64) of the removed duplicates."""
        st = self.stats()
        cap = max(1, int(st["total_rows"]))
        ords = np.empty(cap, dtype=np.uint64)
        ids = np.empty((cap, 16), dtype=np.uint8)
        count = C.c_uint64()
        _ffi.check(_ffi.lib().zb_index_deduplicate(self._h, C.byref(count), ords.ctypes.data, ids.ctypes.data, cap))
        n = int(count.value)
        return ids[:n].copy(), ords[:n].copy()

    # ---------------------------------------------------------------- lsh.rs:506-529, :389-409
    def clear(self) -> None:
        _ffi.check(_ffi.lib().zb_index_clear(self._h))

    def no_vectors(self) -> bool:
        out = C.c_int()
        _ffi.check(_ffi.lib().zb_index_no_vectors(self._h, C.byref(out)))
        return bool(out.value)

    def no_trees(self) -> bool:
        out = C.c_int()
        _ffi.check(_ffi.lib().zb_index_no_trees(self._h, C.byref(out)))
        return bool(out.value)

    def is_empty(self) -> bool:
        return self.no_vectors() or self.no_trees()

    # ---------------------------------------------------------------- lsh.rs:544-565
    # ---------------------------------------------------------------- restricted search (DESIGN 3.10)
    def rowset(self, ids: Optional[Sequence] = None, ordinals=None, exclude: bool = False) -> RowSet:
        """The rows given by `ids` or by `ordinals` (one of the two; duplicates allowed), or with exclude=True every row
        present now except those.  An ordinal at or beyond total_rows raises ZebraError; unknown ids are ignored and reported
        in the RowSet's `found`.  Sharded index: every rank makes it from the same list."""
        if (ids is None) == (ordinals is None):
            raise ValueError("give ids or ordinals")
        flags = ROWSET_EXCLUDE if exclude else 0
        h, count, found = C.c_void_p(), C.c_uint64(), None
        if ids is not None:
            ids = list(ids)
            idb = _ids_to_bytes(ids)
            found = np.zeros(len(ids), dtype=np.uint8)
            _ffi.check(_ffi.lib().zb_index_rowset_from_ids(self._h, len(ids), idb.ctypes.data if ids else None, flags,
                                                           found.ctypes.data, C.byref(count), C.byref(h)))
            found = found.astype(bool)
        else:
            o = np.ascontiguousarray(ordinals, dtype=np.uint64).reshape(-1)
            _ffi.check(_ffi.lib().zb_index_rowset_from_ordinals(self._h, o.size, o.ctypes.data if o.size else None, flags,
                                                                C.byref(count), C.byref(h)))
        rs = RowSet(self, h, int(count.value), found)
        self._rowsets.add(rs)
        return rs

    def _within(self, within: Optional[RowSet]):
        if not isinstance(within, RowSet):
            raise TypeError("within must be a RowSet made by LSHIndex.rowset")
        if within.index is not self:
            raise ValueError("within is a rowset of another index")
        if not within._h.value:   # NULL would be the unrestricted search: a closed set must not widen it
            raise ValueError("within is a closed RowSet")
        return within._h

    # probes (every search form): 0 = the reference's search; P > 0 also visits, in every tree, the leaves across the P
    # main-path planes closest to the query (multi-probe, DESIGN 3.9; at most ZB_MAX_PROBES = 32)
    # within (every search form): a RowSet; the search runs as if every live row outside it had been removed (DESIGN 3.10)
    def search(self, query, top_k: int, metric: Optional[_DeviceMetric] = None, probes: int = 0,
               within: Optional[RowSet] = None) -> List[Tuple[_uuid.UUID, int]]:
        if metric is not None and metric != self.metric:
            raise ValueError("this device index was created for " + type(self.metric).__name__)
        ids, _, bits, counts = self.search_batch(np.asarray(query, np.float32)[None, :], top_k, probes=probes, within=within)
        c = int(counts[0])
        return list(zip(_bytes_to_ids(ids[0, :c]), (int(b) for b in bits[0, :c])))

    def search_batch(self, queries, top_k: int, want_ids: bool = True, probes: int = 0, within: Optional[RowSet] = None):
        """One call for the whole batch (replaces the par_iter of core.rs:299).  Returns
        (ids [nq,k,16] uint8 or None, ordinals [nq,k] uint64, distance bits [nq,k] uint64, counts [nq] uint32)."""
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        nq = q.shape[0]
        ids = np.empty((nq, top_k, 16), dtype=np.uint8) if want_ids else None
        ords = np.empty((nq, top_k), dtype=np.uint64)
        bits = np.empty((nq, top_k), dtype=np.uint64)
        counts = np.zeros(nq, dtype=np.uint32)
        self.search_batch_ptr(nq, q.ctypes.data, top_k, ords.ctypes.data, bits.ctypes.data, counts.ctypes.data,
                              ids.ctypes.data if want_ids else None, probes=probes, within=within)
        return ids, ords, bits, counts

    def search_batch_ptr(self, nq: int, q_ptr: int, top_k: int, ord_ptr: int, bits_ptr: int, counts_ptr: int,
                         ids_ptr: Optional[int] = None, probes: int = 0, within: Optional[RowSet] = None) -> None:
        """Host-pointer form (e.g. pinned buffers owned by the caller)."""
        if within is not None:
            _ffi.check(_ffi.lib().zb_index_search_rowset(self._h, nq, q_ptr, top_k, probes, self._within(within), ids_ptr, ord_ptr,
                                                         bits_ptr, counts_ptr))
        elif probes:
            _ffi.check(_ffi.lib().zb_index_search_probe(self._h, nq, q_ptr, top_k, probes, ids_ptr, ord_ptr, bits_ptr, counts_ptr))
        else:
            _ffi.check(_ffi.lib().zb_index_search_batch(self._h, nq, q_ptr, top_k, ids_ptr, ord_ptr, bits_ptr, counts_ptr))

    def search_batch_device(self, nq: int, d_q_ptr: int, top_k: int, d_ord_ptr: int, d_bits_ptr: int, d_counts_ptr: int,
                            probes: int = 0, within: Optional[RowSet] = None):
        if within is not None:
            _ffi.check(_ffi.lib().zb_index_search_rowset_device(self._h, nq, d_q_ptr, top_k, probes, self._within(within), d_ord_ptr,
                                                                d_bits_ptr, d_counts_ptr))
        elif probes:
            _ffi.check(_ffi.lib().zb_index_search_probe_device(self._h, nq, d_q_ptr, top_k, probes, d_ord_ptr, d_bits_ptr,
                                                               d_counts_ptr))
        else:
            _ffi.check(_ffi.lib().zb_index_search_batch_device(self._h, nq, d_q_ptr, top_k, d_ord_ptr, d_bits_ptr, d_counts_ptr))

    # ---------------------------------------------------------------- exact (brute-force) search, zb_index_search_exact
    def search_exact(self, query, top_k: int, within: Optional[RowSet] = None) -> List[Tuple[_uuid.UUID, int]]:
        """The true top_k over every live row (of `within`, if given), ordered like `search` (ground truth for its recall)."""
        ids, _, bits, counts = self.search_exact_batch(np.asarray(query, np.float32)[None, :], top_k, within=within)
        c = int(counts[0])
        return list(zip(_bytes_to_ids(ids[0, :c]), (int(b) for b in bits[0, :c])))

    def search_exact_batch(self, queries, top_k: int, want_ids: bool = True, within: Optional[RowSet] = None):
        """Returns (ids [nq,k,16] uint8 or None, ordinals [nq,k] uint64, distance bits [nq,k] uint64, counts [nq] uint32).
        Sharded index: collective, every rank passes the same queries and gets the full results."""
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        nq = q.shape[0]
        ids = np.empty((nq, top_k, 16), dtype=np.uint8) if want_ids else None
        ords = np.empty((nq, top_k), dtype=np.uint64)
        bits = np.empty((nq, top_k), dtype=np.uint64)
        counts = np.zeros(nq, dtype=np.uint32)
        if within is not None:
            _ffi.check(_ffi.lib().zb_index_search_exact_rowset(self._h, nq, q.ctypes.data, top_k, self._within(within),
                                                               ids.ctypes.data if want_ids else None, ords.ctypes.data,
                                                               bits.ctypes.data, counts.ctypes.data))
        else:
            _ffi.check(_ffi.lib().zb_index_search_exact(self._h, nq, q.ctypes.data, top_k,
                                                        ids.ctypes.data if want_ids else None, ords.ctypes.data,
                                                        bits.ctypes.data, counts.ctypes.data))
        return ids, ords, bits, counts

    def search_exact_batch_device(self, nq: int, d_q_ptr: int, top_k: int, d_ord_ptr: int, d_bits_ptr: int, d_counts_ptr: int,
                                  within: Optional[RowSet] = None):
        if within is not None:
            _ffi.check(_ffi.lib().zb_index_search_exact_rowset_device(self._h, nq, d_q_ptr, top_k, self._within(within), d_ord_ptr,
                                                                      d_bits_ptr, d_counts_ptr))
        else:
            _ffi.check(_ffi.lib().zb_index_search_exact_device(self._h, nq, d_q_ptr, top_k, d_ord_ptr, d_bits_ptr, d_counts_ptr))

    # ---- sharded index, scalable form: every rank passes (and gets back) only the slice of the batch it fronts ----
    def slice_bounds(self, nq_total: int, shard_rank: int, shard_count: int) -> Tuple[int, int]:
        """Queries [lo, hi) of a batch of nq_total that rank `shard_rank` of `shard_count` fronts (zb_index_search_slice)."""
        nqp = -(-nq_total // max(1, shard_count))
        lo = min(nq_total, shard_rank * nqp)
        return lo, min(nq_total, lo + nqp)

    def search_slice(self, nq_total: int, slice_queries, top_k: int, want_ids: bool = True, probes: int = 0,
                     within: Optional[RowSet] = None):
        """Collective.  `slice_queries` = this rank's slice of the batch; returns that slice's (ids, ordinals, bits, counts)."""
        q = np.ascontiguousarray(slice_queries, dtype=np.float32).reshape(-1, self.dim)
        n = q.shape[0]
        ids = np.empty((n, top_k, 16), dtype=np.uint8) if want_ids else None
        ords = np.empty((n, top_k), dtype=np.uint64)
        bits = np.empty((n, top_k), dtype=np.uint64)
        counts = np.zeros(n, dtype=np.uint32)
        self.search_slice_ptr(nq_total, q.ctypes.data if n else None, top_k, ords.ctypes.data if n else None,
                              bits.ctypes.data if n else None, counts.ctypes.data if n else None,
                              ids.ctypes.data if want_ids and n else None, probes=probes, within=within)
        return ids, ords, bits, counts

    def search_slice_ptr(self, nq_total: int, q_ptr: int, top_k: int, ord_ptr: int, bits_ptr: int, counts_ptr: int,
                         ids_ptr: Optional[int] = None, probes: int = 0, within: Optional[RowSet] = None) -> None:
        if within is not None:
            _ffi.check(_ffi.lib().zb_index_search_slice_rowset(self._h, nq_total, q_ptr, top_k, probes, self._within(within), ids_ptr,
                                                               ord_ptr, bits_ptr, counts_ptr))
        elif probes:
            _ffi.check(_ffi.lib().zb_index_search_slice_probe(self._h, nq_total, q_ptr, top_k, probes, ids_ptr, ord_ptr, bits_ptr,
                                                              counts_ptr))
        else:
            _ffi.check(_ffi.lib().zb_index_search_slice(self._h, nq_total, q_ptr, top_k, ids_ptr, ord_ptr, bits_ptr, counts_ptr))

    def search_prefetch_ptr(self, n: int, q_ptr: int):
        """Announce the next batch (zb_index_search_prefetch): its upload overlaps the search call in between."""
        _ffi.check(_ffi.lib().zb_index_search_prefetch(self._h, n, q_ptr))

    def search_slice_device(self, nq_total: int, d_q_ptr: int, top_k: int, d_ord_ptr: int, d_bits_ptr: int, d_counts_ptr: int,
                            probes: int = 0, within: Optional[RowSet] = None):
        if within is not None:
            _ffi.check(_ffi.lib().zb_index_search_slice_rowset_device(self._h, nq_total, d_q_ptr, top_k, probes, self._within(within),
                                                                      d_ord_ptr, d_bits_ptr, d_counts_ptr))
        elif probes:
            _ffi.check(_ffi.lib().zb_index_search_slice_probe_device(self._h, nq_total, d_q_ptr, top_k, probes, d_ord_ptr,
                                                                     d_bits_ptr, d_counts_ptr))
        else:
            _ffi.check(_ffi.lib().zb_index_search_slice_device(self._h, nq_total, d_q_ptr, top_k, d_ord_ptr, d_bits_ptr, d_counts_ptr))

    # ---------------------------------------------------------------- bucket keys
    def hash(self, rows):
        x = np.ascontiguousarray(rows, dtype=np.float32).reshape(-1, self.dim)
        n, t = x.shape[0], self.options.num_trees
        keys = np.zeros((n, t), dtype=np.uint64)
        depth = np.zeros((n, t), dtype=np.uint32)
        leaf = np.zeros((n, t), dtype=np.int32)
        _ffi.check(_ffi.lib().zb_index_hash(self._h, n, x.ctypes.data, keys.ctypes.data, depth.ctypes.data, leaf.ctypes.data))
        return keys, depth, leaf

    def hash_device(self, n: int, d_rows_ptr: int, d_keys_ptr: int, d_depth_ptr: int = 0, d_leaf_ptr: int = 0):
        _ffi.check(_ffi.lib().zb_index_hash_device(self._h, n, d_rows_ptr, d_keys_ptr or None, d_depth_ptr or None,
                                                   d_leaf_ptr or None))

    # ---------------------------------------------------------------- forest interchange
    def export_forest(self) -> Forest:
        sz = np.zeros(4, dtype=np.int64)
        _ffi.check(_ffi.lib().zb_index_forest_sizes(self._h, sz.ctypes.data))
        nn, npl, nl, nm = (int(v) for v in sz)
        nodes = np.zeros((nn, 4), dtype=np.int32)
        roots = np.zeros(self.options.num_trees, dtype=np.int32)
        coef = np.zeros((npl, self.dim), dtype=np.float32)
        cst = np.zeros(npl, dtype=np.float32)
        leaf_off = np.zeros(nl + 1, dtype=np.int64)
        members = np.zeros(nm, dtype=np.uint64)
        _ffi.check(_ffi.lib().zb_index_export_forest(self._h, nodes.ctypes.data, roots.ctypes.data, coef.ctypes.data,
                                                     cst.ctypes.data, leaf_off.ctypes.data, members.ctypes.data))
        return Forest(nodes, roots, coef, cst, leaf_off, members)

    def load_forest(self, rows, forest, ids: Optional[Sequence] = None) -> None:
        rows = np.ascontiguousarray(rows, dtype=np.float32).reshape(-1, self.dim)
        f = Forest(forest.nodes, forest.roots, forest.coef, forest.cst, forest.leaf_off, forest.members)
        sz = np.array([f.nodes.shape[0], f.cst.shape[0], f.leaf_off.shape[0] - 1, f.members.shape[0]], dtype=np.int64)
        idb = _ids_to_bytes(ids) if ids is not None else None
        _ffi.check(_ffi.lib().zb_index_load_forest(self._h, rows.shape[0], rows.ctypes.data,
                                                   idb.ctypes.data if idb is not None else None, sz.ctypes.data,
                                                   f.nodes.ctypes.data, f.roots.ctypes.data, f.coef.ctypes.data,
                                                   f.cst.ctypes.data, f.leaf_off.ctypes.data, f.members.ctypes.data))

    def load_flat(self, rows, bits: int, coef, cst, ids: Optional[Sequence] = None) -> None:
        """FLAT tables (the K-bit LSH table of north_star (a)): every node at depth d of tree t shares plane
        ``coef[t * bits + d]``.  The rows are bucketed by one dense projection on the device (sign bits packed into the keys
        with __ballot_sync); the index then holds the equivalent forest of complete trees."""
        rows = np.ascontiguousarray(rows, dtype=np.float32).reshape(-1, self.dim)
        h = self.options.num_trees * int(bits)
        coef = np.ascontiguousarray(coef, dtype=np.float32).reshape(h, self.dim)
        cst = np.ascontiguousarray(cst, dtype=np.float32).reshape(h)
        idb = _ids_to_bytes(ids) if ids is not None else None
        _ffi.check(_ffi.lib().zb_index_load_flat(self._h, rows.shape[0], rows.ctypes.data,
                                                 idb.ctypes.data if idb is not None else None, int(bits), coef.ctypes.data,
                                                 cst.ctypes.data))

    # ---------------------------------------------------------------- the reference's stored values (SURVEY 8f row 4)
    def import_store(self, ids: Sequence, embeddings, tree_blobs: Sequence[bytes]) -> dict:
        """Replace the index content with a reference store: the (key, value) pairs of the `embeddings` partition
        (lsh.rs:91-97) and the values of the `trees` partition (lsh.rs:99-105).  Returns the import report plus
        ``orphans`` (ids of embeddings some tree did not hold; they are NOT loaded -- re-insert them with add())."""
        rows = np.ascontiguousarray(embeddings, dtype=np.float32).reshape(-1, self.dim)
        idb = ids if isinstance(ids, np.ndarray) else _ids_to_bytes(ids)
        idb = np.ascontiguousarray(idb, dtype=np.uint8).reshape(-1)
        n = rows.shape[0]
        if idb.size != 16 * n:
            raise ValueError("ids must hold one 16-byte id per row")
        bufs = [np.frombuffer(bytes(b), dtype=np.uint8) for b in tree_blobs]
        ptrs = (C.c_void_p * max(1, len(bufs)))(*[b.ctypes.data for b in bufs])
        sizes = np.array([b.size for b in bufs] or [0], dtype=np.uint64)
        rep = _ffi.ImportReport()
        orphans = np.zeros((max(1, n), 16), dtype=np.uint8)
        _ffi.check(_ffi.lib().zb_index_import_store(self._h, n, idb.ctypes.data if n else None, rows.ctypes.data if n else None,
                                                    len(bufs), ptrs, sizes.ctypes.data, C.byref(rep), orphans.ctypes.data, n))
        out = rep.as_dict()
        out["orphans"] = _bytes_to_ids(orphans[: int(rep.orphan_rows)])
        return out

    def export_rows(self, first_ordinal: int = 0, n: Optional[int] = None):
        """(embeddings [n,dim] f32, ids [n,16] uint8, live [n] bool) of ordinals [first, first + n) -- unsharded index."""
        if n is None:
            n = int(self.stats()["total_rows"]) - first_ordinal
        rows = np.zeros((n, self.dim), dtype=np.float32)
        ids = np.zeros((n, 16), dtype=np.uint8)
        live = np.zeros(n, dtype=np.uint8)
        _ffi.check(_ffi.lib().zb_index_export_rows(self._h, first_ordinal, n, rows.ctypes.data, ids.ctypes.data, live.ctypes.data))
        return rows, ids, live.astype(bool)

    def export_tree_blobs(self) -> List[bytes]:
        """Every tree as the reference's `trees` value (bincode(legacy) Node<N>); removed rows are left out of the leaves.
        One export of the forest serves all trees (zb_index_export_tree_blobs)."""
        t = self.options.num_trees
        sizes = np.zeros(t, dtype=np.uint64)
        total = C.c_uint64()
        _ffi.check(_ffi.lib().zb_index_export_tree_blobs(self._h, None, 0, sizes.ctypes.data, C.byref(total)))
        buf = np.empty(max(1, int(total.value)), dtype=np.uint8)
        _ffi.check(_ffi.lib().zb_index_export_tree_blobs(self._h, buf.ctypes.data, int(total.value), sizes.ctypes.data, C.byref(total)))
        out, at = [], 0
        for n in sizes:
            out.append(buf[at:at + int(n)].tobytes())
            at += int(n)
        return out

    def export_tree_blob(self, tree: int) -> bytes:
        need = C.c_uint64()
        _ffi.check(_ffi.lib().zb_index_export_tree_blob(self._h, tree, None, 0, C.byref(need)))
        buf = np.empty(int(need.value), dtype=np.uint8)
        _ffi.check(_ffi.lib().zb_index_export_tree_blob(self._h, tree, buf.ctypes.data, buf.size, C.byref(need)))
        return buf.tobytes()

    def save_store(self, path: str, zebra: bytes = b"") -> None:
        """Dump both partitions (live rows only, as the reference deletes removed keys) into one file, see interchange.py."""
        from . import interchange

        rows, ids, live = self.export_rows()
        blobs = self.export_tree_blobs() if not self.no_trees() else []
        interchange.write_store(path, self.dim, zebra, [(interchange.tree_key(t), b) for t, b in enumerate(blobs)],
                                ids[live], rows[live])

    def load_store(self, path: str) -> dict:
        from . import interchange

        dim, _, trees, ids, rows = interchange.read_store(path)
        if dim != self.dim:
            raise ValueError(f"store holds {dim}-dimensional vectors, this index {self.dim}")
        if not trees:
            self.clear()
            if rows.shape[0]:
                self.add(rows, ids.reshape(-1, 16))
            return {"rows_loaded": int(rows.shape[0]), "orphans": []}
        return self.import_store(ids, rows, [b for _, b in trees])

    # ---------------------------------------------------------------- misc
    def stats(self) -> dict:
        st = _ffi.Stats()
        _ffi.check(_ffi.lib().zb_index_stats(self._h, C.byref(st)))
        return st.as_dict()

    def stream_ptr(self) -> int:
        """cudaStream_t of the index (all kernels are launched on it)."""
        out = C.c_void_p()
        _ffi.check(_ffi.lib().zb_index_stream(self._h, C.byref(out)))
        return int(out.value or 0)

    def set_param(self, key: str, value: int) -> None:
        _ffi.check(_ffi.lib().zb_index_set_param(self._h, key.encode(), int(value)))

    def comm_init(self, unique_id: bytes) -> None:
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        _ffi.check(_ffi.lib().zb_index_comm_init(self._h, buf))


def recall_at_k(approx_ords, approx_counts, exact_ords, exact_counts) -> np.ndarray:
    """Per query |approx ∩ exact| / count(exact) over the first counts[q] ordinals of each [nq, k] list; 1.0 where the
    exact list is empty."""
    a = np.asarray(approx_ords, dtype=np.uint64)
    e = np.asarray(exact_ords, dtype=np.uint64)
    ac = np.asarray(approx_counts).astype(np.int64).reshape(-1)
    ec = np.asarray(exact_counts).astype(np.int64).reshape(-1)
    out = np.ones(ec.shape[0], dtype=np.float64)
    for q in range(ec.shape[0]):
        if ec[q]:
            out[q] = np.intersect1d(a[q, :ac[q]], e[q, :ec[q]]).size / ec[q]
    return out


def comm_unique_id() -> bytes:
    buf = (C.c_uint8 * 128)()
    _ffi.check(_ffi.lib().zb_comm_unique_id(buf))
    return bytes(buf)


def synth_fill_device(device: int, d_ptr: int, first_row: int, row_stride: int, n: int, dim: int, seed: int, kind: int = 0):
    _ffi.check(_ffi.lib().zb_synth_fill_device(device, d_ptr, first_row, row_stride, n, dim, seed, kind))
