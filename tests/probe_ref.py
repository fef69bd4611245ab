"""The multi-probe search rule (DESIGN 3.9, include/zebra_b200.h) stated on top of the CPU oracle.  TEST INFRASTRUCTURE ONLY.

Multi-probe search is this project's extension, not part of the reference, so it is not in oracle/ (the restatement of the
reference).  ProbeOracle wraps an oracle.zb_oracle.OracleIndex and keeps the rows and tombstones it was given:

* the cascade of every tree is the oracle's own (`candidates` / `trace`), unchanged;
* the main path's margin keys use the oracle's canonical dot (zbo_dot_f32) and its point_is_above;
* each probe leaf contributes its min(live, top_k) nearest live rows by (distance bits, id), the oracle's distance bits;
* the union is rescored and ordered like zbo_search.

With probes = 0 every method returns the oracle's own result.  tests/test_probe_oracle.py pins this module against a second,
pure-Python restatement on tests/pyref.py's exact-rational arithmetic and against a hand-built known-answer forest.
"""
from __future__ import annotations

import math
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from oracle import zb_oracle as zo

SENT = np.iinfo(np.uint64).max


def probe_key(coef, cst, q) -> float:
    """|v| / sqrt(n2), v = (f64)dot(coef, q) + (f64)cst, n2 = (f64)dot(coef, coef); +inf for a NaN v, n2 of 0 or not finite."""
    v = zo.dot(coef, q) + float(np.float32(cst))
    n2 = zo.dot(coef, coef)
    if math.isnan(v) or not n2 > 0.0 or math.isinf(n2):
        return math.inf
    return abs(v) / math.sqrt(n2)


class ProbeOracle:
    def __init__(self, dim: int, metric: int, max_node_size: int = 5, num_trees: int = 15, seed: int = 0):
        self.dim, self.metric = dim, metric
        self.orc = zo.OracleIndex(dim, metric, max_node_size, num_trees, seed)
        self.rows = np.zeros((0, dim), np.float32)
        self.tomb = np.zeros(0, bool)
        self._forest = None

    # ---- mutations: forwarded to the oracle, mirrored here
    def add(self, rows):
        rows = np.ascontiguousarray(rows, np.float32).reshape(-1, self.dim)
        ids = self.orc.add(rows)
        self.rows = np.concatenate([self.rows, rows])
        self.tomb = np.concatenate([self.tomb, np.zeros(rows.shape[0], bool)])
        self._forest = None
        return ids

    def remove(self, ids):
        ids = np.ascontiguousarray(ids, np.uint64)
        done = self.orc.remove(ids)
        self.tomb[ids[done].astype(np.int64)] = True
        return done

    def load_forest(self, rows, forest):
        self.orc.load_forest(rows, forest)
        self.rows = np.ascontiguousarray(rows, np.float32).reshape(-1, self.dim).copy()
        self.tomb = np.zeros(self.rows.shape[0], bool)
        self._forest = None

    def export_forest(self):
        return self.orc.export_forest()

    @property
    def forest(self):
        if self._forest is None:
            self._forest = self.orc.export_forest()
        return self._forest

    # ---- the probe rule
    def _live(self, leaf):
        f = self.forest
        m = f.members[int(f.leaf_off[leaf]):int(f.leaf_off[leaf + 1])].astype(np.int64)
        return m[~self.tomb[m]]

    def probe_leaves(self, q, probes):
        """Per tree, the probe leaves in the order they are picked."""
        f = self.forest
        out = []
        for root in f.roots:
            path, node, depth = [], int(root), 0
            while f.nodes[node][0] >= 0:   # the main path: the walk's first root-to-leaf descent
                plane, left, right, _ = (int(v) for v in f.nodes[node])
                above = zo.point_is_above(f.coef[plane], float(f.cst[plane]), q)
                path.append((probe_key(f.coef[plane], f.cst[plane], q), depth, left if above else right))
                node, depth = (right if above else left), depth + 1
            leaves = []
            for _, _, node in sorted(path)[:probes]:
                while f.nodes[node][0] >= 0:   # greedy descent of the backup side
                    plane, left, right, _ = (int(v) for v in f.nodes[node])
                    node = right if zo.point_is_above(f.coef[plane], float(f.cst[plane]), q) else left
                leaves.append(int(f.nodes[node][3]))
            out.append(leaves)
        return out

    def _bits(self, ids, q):
        if not ids.size:
            return np.zeros(0, np.uint64)
        return zo.distance_bits_batch(self.metric, self.rows[ids], np.broadcast_to(q, (ids.size, self.dim)))

    def search(self, query, top_k: int, probes: int = 0):
        q = np.ascontiguousarray(query, np.float32)
        if not probes:
            return self.orc.search(q, top_k)
        cand = [self.orc.candidates(q, top_k).astype(np.int64)]
        if self.orc.num_rows and top_k:
            for leaves in self.probe_leaves(q, probes):
                for leaf in leaves:
                    live = self._live(leaf)
                    if live.size:   # a visit with n' = top_k: the top_k nearest live rows by (bits, id)
                        order = np.lexsort((live, self._bits(live, q)))[:top_k]
                        cand.append(live[order])
        ids = np.unique(np.concatenate(cand))
        bits = self._bits(ids, q)
        order = np.lexsort((ids, bits))[:top_k]
        return ids[order].astype(np.uint64), bits[order]

    def search_batch(self, queries, top_k: int, nthreads: int = 1, probes: int = 0):
        q = np.ascontiguousarray(queries, np.float32).reshape(-1, self.dim)
        if not probes:
            return self.orc.search_batch(q, top_k, nthreads=nthreads)
        nq = q.shape[0]
        ids = np.full((nq, max(top_k, 1)), SENT, np.uint64)
        bits = np.full((nq, max(top_k, 1)), SENT, np.uint64)
        counts = np.zeros(nq, np.uint32)
        _ = self.forest   # export once, before the threads read it
        with ThreadPoolExecutor(max(1, nthreads)) as ex:
            for i, (o, b) in enumerate(ex.map(lambda x: self.search(x, top_k, probes), q)):
                ids[i, :o.size], bits[i, :o.size], counts[i] = o, b, o.size
        return ids[:, :top_k], bits[:, :top_k], counts

    def trace(self, query, top_k: int, probes: int = 0) -> np.ndarray:
        """The oracle's visit plan, each tree's probe visits (tree, leaf, top_k, live) after its cascade."""
        q = np.ascontiguousarray(query, np.float32)
        tr = self.orc.trace(q, top_k)
        if not probes or not self.orc.num_rows:
            return tr
        rows = []
        for t, leaves in enumerate(self.probe_leaves(q, probes)):
            rows += tr[tr[:, 0] == t].tolist()
            rows += [[t, leaf, top_k, int(self._live(leaf).size)] for leaf in leaves]
        return np.array(rows, np.int32).reshape(-1, 4)
