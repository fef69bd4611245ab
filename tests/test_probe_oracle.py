"""Multi-probe search (DESIGN 3.9) in the CPU reference: tests/probe_ref.py (the probe rule over the C oracle) against a
second, pure-Python restatement on tests/pyref.py's arithmetic, a known-answer forest, and the properties the GPU tests rely
on."""
import math

import numpy as np
import pytest

import pyref
from oracle import zb_oracle as zo
from probe_ref import ProbeOracle


def _dot(a, b) -> float:
    """The canonical f32 dot widened to f64, NaN when an input is NaN (pyref's rational emulation takes finite values)."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    if np.isnan(a).any() or np.isnan(b).any():
        return math.nan
    return float(pyref.dot16(a, b))


def _above(coef, cst, q) -> bool:
    return _dot(coef, q) + float(cst) >= 0.0   # NaN is below


def probe_key(coef, cst, q) -> float:
    v = _dot(coef, q) + float(np.float32(cst))
    n2 = _dot(coef, coef)
    if math.isnan(v) or not n2 > 0.0 or math.isinf(n2):
        return math.inf
    return abs(v) / math.sqrt(n2)


def py_probe_search(py, q, top_k, probes):
    """search with `probes` probe leaves per tree, restated from the rule in include/zebra_b200.h."""
    nodes = py.f.nodes
    cand, trace = set(), []
    for t, root in enumerate(py.f.roots):
        py.tree_result(q, top_k, int(root), cand, trace, t)
        path, node, depth = [], int(root), 0
        while nodes[node][0] >= 0:   # the main path: the walk's first root-to-leaf descent
            plane, left, right, _ = (int(v) for v in nodes[node])
            above = _above(py.f.coef[plane], py.f.cst[plane], q)
            path.append((probe_key(py.f.coef[plane], py.f.cst[plane], q), depth, left if above else right))
            node, depth = (right if above else left), depth + 1
        for _, _, node in sorted(path)[:probes]:
            while nodes[node][0] >= 0:
                plane, left, right, _ = (int(v) for v in nodes[node])
                node = right if _above(py.f.coef[plane], py.f.cst[plane], q) else left
            py.tree_result(q, top_k, node, cand, trace, t)
    scored = sorted((py.dist_bits(py.rows[i], q), i) for i in cand)
    return scored[:top_k], trace


def _pyforest(ix, rows, tomb):
    return pyref.PyForest(ix.export_forest(), rows, tomb, lambda r, q: zo.distance_bits(ix.metric, r, q), _above)


def _check(ix, py, q, k, probes):
    ids, bits = ix.search(q, k, probes=probes)
    exp, trace = py_probe_search(py, q, k, probes)
    assert ids.tolist() == [i for _, i in exp]
    assert bits.tolist() == [b for b, _ in exp]
    assert [tuple(r) for r in ix.trace(q, k, probes=probes).tolist()] == trace
    return trace


def full_tree(rows, depth, plane_of):
    """One tree of the given depth; plane_of(path) -> (coef, cst) for the inner node at that sign path (0 = below).  Rows go
    to the leaf point_is_above sends them to; leaves are numbered in preorder (leaf of path p = int(p, 2))."""
    nodes, coef, cst, leaf_off, members = [], [], [], [0], []

    def route(x):
        p = ()
        while len(p) < depth:
            c, k = plane_of(p)
            p += (int(zo.point_is_above(c, k, x)),)
        return p

    routes = [route(x) for x in rows]

    def rec(path):
        me = len(nodes)
        nodes.append(None)
        if len(path) == depth:
            members.extend(i for i, r in enumerate(routes) if r == path)
            nodes[me] = [-1, -1, -1, len(leaf_off) - 1]
            leaf_off.append(len(members))
        else:
            c, k = plane_of(path)
            pl = len(coef)
            coef.append(np.asarray(c, np.float32))
            cst.append(k)
            left = rec(path + (0,))
            right = rec(path + (1,))
            nodes[me] = [pl, left, right, -1]
        return me

    rec(())
    return zo.Forest(nodes, [0], np.stack(coef), cst, leaf_off, members)


def _axis(dim, i, scale=1.0):
    c = np.zeros(dim, np.float32)
    c[i] = scale
    return c


# ---------------------------------------------------------------------------------------------------- restatement
@pytest.mark.parametrize("metric", [zo.COSINE, zo.L2SQ, zo.L2, zo.MANHATTAN])
@pytest.mark.parametrize("mns,trees,k", [(5, 6, 10), (3, 3, 4), (32, 4, 10), (64, 2, 3)])
def test_c_probe_equals_python_restatement(metric, mns, trees, k):
    rng = np.random.default_rng(mns * 31 + trees + metric)
    dim, n = 20, 300
    rows = rng.standard_normal((n, dim)).astype(np.float32)
    ix = ProbeOracle(dim, metric, max_node_size=mns, num_trees=trees, seed=3)
    ix.add(rows)
    dead = rng.choice(n, 40, replace=False)
    ix.remove(dead)
    tomb = np.zeros(n, dtype=bool)
    tomb[dead] = True
    py = _pyforest(ix, rows, tomb)
    qs = np.concatenate([rng.standard_normal((3, dim)).astype(np.float32), rows[:2]])
    for q in qs:
        for probes in (0, 1, 2, 5, 40):   # 40: above every path length here
            trace = _check(ix, py, q, k, probes)
            if probes == 0:
                assert [tuple(r) for r in ix.trace(q, k).tolist()] == trace


def edge_forest(dim=16):
    """Depth 3.  Root: x0 >= 0.  Depth 1: 2 x1 >= 0.  Depth 2: x2 >= 0, except the node at path (1, 1), a zero plane with
    constant 0.5 (always above, key +inf; its below leaf is empty)."""
    def plane_of(p):
        if len(p) == 0:
            return _axis(dim, 0), 0.0
        if len(p) == 1:
            return _axis(dim, 1, 2.0), 0.0
        if p == (1, 1):
            return np.zeros(dim, np.float32), 0.5
        return _axis(dim, 2), 0.0

    rng = np.random.default_rng(7)
    rows = rng.standard_normal((40, dim)).astype(np.float32)
    return full_tree(rows, 3, plane_of), rows


@pytest.mark.parametrize("metric", [zo.L2SQ, zo.COSINE])
def test_edge_cases_match_restatement(metric):
    dim = 16
    forest, rows = edge_forest(dim)
    ix = ProbeOracle(dim, metric, max_node_size=8, num_trees=1)
    ix.load_forest(rows, forest)
    ix.remove([3, 11])
    tomb = np.zeros(rows.shape[0], dtype=bool)
    tomb[[3, 11]] = True
    py = _pyforest(ix, rows, tomb)

    def q_of(x0, x1, x2):
        q = np.zeros(dim, np.float32)
        q[:3] = (x0, x1, x2)
        return q

    on_plane = q_of(0.0, -0.25, 3.0)     # v = 0 at the root: key 0, above
    tied = q_of(-2.0, 0.5, -0.5)         # depth 1: |2 * 0.5| / 2 = 0.5, depth 2: |-0.5| / 1 = 0.5 -- the shallower first
    zero_plane = q_of(1.0, 1.0, 0.1)     # path (1, 1): the zero plane, key +inf
    nan_q = q_of(np.nan, 1.0, 1.0)       # every v NaN: keys +inf, every side below
    for k in (1, 3, 12):                 # 12: the leaves hold fewer rows, the cascade runs
        for q in (on_plane, tied, zero_plane, nan_q):
            for probes in range(5):      # 4 is above the path length
                _check(ix, py, q, k, probes)
    assert probe_key(_axis(dim, 0), 0.0, on_plane) == 0.0
    assert probe_key(_axis(dim, 1, 2.0), 0.0, tied) == probe_key(_axis(dim, 2), 0.0, tied) == 0.5
    assert probe_key(np.zeros(dim, np.float32), 0.5, zero_plane) == math.inf
    assert probe_key(_axis(dim, 0), 0.0, nan_q) == math.inf
    # the tie: at P = 1 the depth-1 node is flipped, not the depth-2 one
    tr1 = ix.trace(tied, 1, probes=1).tolist()
    main = ix.trace(tied, 1).tolist()
    assert tr1[: len(main)] == main
    # tied's main leaf: x0 < 0, 2 x1 >= 0, x2 < 0 -> path (0, 1, 0) = leaf 2; flipping depth 1 -> (0, 0, .) with x2 < 0 -> leaf 0
    assert main[0][1] == 2 and tr1[-1][1] == 0


# ---------------------------------------------------------------------------------------------------- known answer
def kat_depth3(dim=4):
    """Axis planes x0, x1, x2 (constant 0) at depths 0, 1, 2; leaf (a0 a1 a2) (1 = above) = 4 a0 + 2 a1 + a2 holds three
    rows with that sign pattern: ids 3 * leaf + j."""
    rows = np.zeros((24, dim), np.float32)
    for leaf in range(8):
        s = [1.0 if (leaf >> (2 - b)) & 1 else -1.0 for b in range(3)]
        for j in range(3):
            rows[3 * leaf + j, :3] = [v * (1 + j) for v in s]
            rows[3 * leaf + j, 3] = j
    forest = full_tree(rows, 3, lambda p: (_axis(dim, len(p)), 0.0))
    assert forest.members.tolist() == list(range(24))
    return forest, rows


def test_known_answer_forest():
    forest, rows = kat_depth3()
    ix = ProbeOracle(4, zo.L2SQ, max_node_size=3, num_trees=1)
    ix.load_forest(rows, forest)
    q = np.array([0.3, -0.1, 2.0, 0.0], np.float32)
    # main path: above, below, above -> leaf 5.  Keys by depth: 0.3, 0.1, 2.0 -> flips in the order depth 1, 0, 2:
    # depth 1 -> (1, 1, 1) = leaf 7; depth 0 -> (0, 0, 1) = leaf 1; depth 2 -> (1, 0, 0) = leaf 4
    expect = {0: [5], 1: [5, 7], 2: [5, 7, 1], 3: [5, 7, 1, 4], 4: [5, 7, 1, 4]}
    for probes, leaves in expect.items():
        assert ix.trace(q, 2, probes=probes).tolist() == [[0, leaf, 2, 3] for leaf in leaves]
    ids, _ = ix.search(q, 2, probes=0)
    assert set(ids.tolist()) <= {15, 16, 17}
    # a probe leaf without live rows is listed, contributes nothing and is not replaced by another leaf
    ix.remove([21, 22, 23])
    assert ix.trace(q, 2, probes=1).tolist() == [[0, 5, 2, 3], [0, 7, 2, 0]]
    ids, _ = ix.search(q, 3, probes=1)   # leaf 5 fills the budget: no cascade, and the empty probe leaf adds nothing
    assert sorted(ids.tolist()) == [15, 16, 17]
    assert ix.trace(q, 3, probes=1).tolist() == [[0, 5, 3, 3], [0, 7, 3, 0]]


# ---------------------------------------------------------------------------------------------------- properties
def _brute(rows, tomb, metric, q, k):
    live = np.flatnonzero(~tomb)
    bits = zo.distance_bits_batch(metric, rows[live], np.broadcast_to(q, (live.size, q.size)))
    order = sorted(zip(bits.tolist(), live.tolist()))[:k]
    return [i for _, i in order], [b for b, _ in order]


def test_probes_zero_is_the_reference_search():
    rng = np.random.default_rng(1)
    dim, n, k = 24, 2000, 10
    rows = rng.standard_normal((n, dim)).astype(np.float32)
    ix = ProbeOracle(dim, zo.L2, max_node_size=16, num_trees=3, seed=2)
    ix.add(rows)
    plain = zo.OracleIndex(dim, zo.L2, max_node_size=16, num_trees=3, seed=2)
    plain.add(rows)
    qs = rng.standard_normal((50, dim)).astype(np.float32)
    for x, y in zip(plain.search_batch(qs, k, nthreads=2), ix.search_batch(qs, k, nthreads=2, probes=0)):
        assert np.array_equal(x, y)
    for q in qs[:10]:
        for x, y in zip(plain.search(q, k), ix.search(q, k, probes=0)):
            assert np.array_equal(x, y)
        assert np.array_equal(plain.trace(q, k), ix.trace(q, k, probes=0))
        # P = 1 ranks a superset of P = 0's candidates: every position of its list is at least as near
        _, bits0 = ix.search(q, k, probes=0)
        _, bits1 = ix.search(q, k, probes=1)
        assert bits1.size >= bits0.size and (bits1[:bits0.size] <= bits0).all()


@pytest.mark.parametrize("metric", [zo.L2SQ, zo.COSINE])
def test_recall_never_falls_as_probes_grow(metric):
    rng = np.random.default_rng(2)
    dim, n, k = 32, 3000, 10
    centres = rng.standard_normal((12, dim)).astype(np.float32)
    rows = (centres[rng.integers(0, 12, n)] + 0.3 * rng.standard_normal((n, dim))).astype(np.float32)
    ix = ProbeOracle(dim, metric, max_node_size=64, num_trees=2, seed=4)
    ix.add(rows)
    dead = rng.choice(n, 300, replace=False)
    ix.remove(dead)
    tomb = np.zeros(n, dtype=bool)
    tomb[dead] = True
    qs = (centres[rng.integers(0, 12, 40)] + 0.3 * rng.standard_normal((40, dim))).astype(np.float32)
    truth = [set(_brute(rows, tomb, metric, q, k)[0]) for q in qs]
    prev, totals = None, []
    for probes in (0, 1, 2, 4, 8):
        ids, _, counts = ix.search_batch(qs, k, nthreads=2, probes=probes)
        found = [set(ids[i, : counts[i]].tolist()) & truth[i] for i in range(len(qs))]
        if prev is not None:
            assert all(p <= f for p, f in zip(prev, found))   # every true top-k row found at P is still found
        prev = found
        totals.append(sum(len(f) for f in found))
    assert totals[-1] > totals[0]


@pytest.mark.parametrize("metric", [zo.COSINE, zo.L2SQ, zo.L2, zo.MANHATTAN])
def test_single_plane_trees_with_a_probe_are_exact(metric):
    rng = np.random.default_rng(3)
    dim, n, trees = 20, 500, 3
    rows = rng.standard_normal((n, dim)).astype(np.float32)
    # T trees, each one plane through two rows with two leaves
    fs = [full_tree(rows, 1, lambda p, t=t: zo.make_plane(rows[2 * t], rows[2 * t + 1])) for t in range(trees)]
    nodes, coef, cst, leaf_off, members, roots = [], [], [], [0], [], []
    for f in fs:
        base_n, base_p, base_l = len(nodes), len(coef), len(leaf_off) - 1
        roots.append(base_n)
        for nd in f.nodes.tolist():
            nodes.append([nd[0] + base_p if nd[0] >= 0 else -1, nd[1] + base_n if nd[1] >= 0 else -1,
                          nd[2] + base_n if nd[2] >= 0 else -1, nd[3] + base_l if nd[3] >= 0 else -1])
        coef.extend(f.coef)
        cst.extend(f.cst.tolist())
        members.extend(f.members.tolist())
        leaf_off.extend((f.leaf_off[1:] + leaf_off[-1]).tolist())
    forest = zo.Forest(nodes, roots, np.stack(coef), cst, leaf_off, members)
    ix = ProbeOracle(dim, metric, max_node_size=n, num_trees=trees)
    ix.load_forest(rows, forest)
    dead = rng.choice(n, 50, replace=False)
    ix.remove(dead)
    tomb = np.zeros(n, dtype=bool)
    tomb[dead] = True
    for q in rng.standard_normal((12, dim)).astype(np.float32):
        for k in (1, 10, 100):
            ids, bits = ix.search(q, k, probes=1)
            eids, ebits = _brute(rows, tomb, metric, q, k)
            assert ids.tolist() == eids and bits.tolist() == ebits
