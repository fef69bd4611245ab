"""Multi-probe search on the GPU (zb_index_search_probe*, DESIGN 3.9): every result field bit for bit against the probe rule
over the CPU oracle (tests/probe_ref.py) across metrics, dims, k, probes, leaf sizes and scan paths; P = 0 against the plain calls; single-plane
trees against the exact search; recall monotone in P; stats, entry-point agreement and errors."""
import numpy as np
import pytest

from oracle import zb_oracle as zo
from probe_ref import ProbeOracle

pytestmark = pytest.mark.gpu

F32 = np.float32
KS = [1, 10, 16, 17, 32, 33, 100, 128, 129]
PS = [1, 2, 5, 32]
# metric code -> (class name, constructor args)
METRICS = {zo.COSINE: ("CosineDistance", ()), zo.L2SQ: ("L2SquaredDistance", ()), zo.L2: ("L2Distance", ()),
           zo.MANHATTAN: ("ManhattanDistance", ()), zo.HAMMING: ("HammingDistance", ()),
           zo.MINKOWSKI(3): ("MinkowskiDistance", (3,))}


def zb():
    import zebra_b200

    return zebra_b200


def clustered(rng, n, dim, centres=24, noise=0.25):
    c = rng.standard_normal((centres, dim)).astype(F32)
    return (c[rng.integers(0, centres, n)] + noise * rng.standard_normal((n, dim))).astype(F32)


def pair(metric, dim, rows, mns, trees, seed=3, load=True):
    """(oracle, device index) over the same forest: the oracle's, loaded (load=True), or both built from `rows`."""
    z = zb()
    name, args = METRICS[metric]
    orc = ProbeOracle(dim, metric, mns, trees, seed=seed)
    orc.add(rows)
    ix = z.LSHIndex(dim, z.LSHIndexOptions(mns, trees), getattr(z, name)(*args), seed=seed)
    if load:
        ix.load_forest(rows, orc.export_forest())
    else:
        ix.add(rows)
    return orc, ix


def parity(orc, ix, qs, k, probes, what=""):
    ids, o, b, c = ix.search_batch(qs, k, probes=probes)
    eo, eb, ec = orc.search_batch(qs, k, nthreads=8, probes=probes)
    assert np.array_equal(c, ec), (what, k, probes)
    assert np.array_equal(o, eo), (what, k, probes)
    assert np.array_equal(b, eb), (what, k, probes)
    for q in range(qs.shape[0]):
        assert (ids[q, c[q]:] == 0xFF).all()
    return o, b, c


def _stats(ix):
    return {k: v for k, v in ix.stats().items() if not k.startswith("last_ms")}


# ---------------------------------------------------------------- P = 0 is the plain call
def test_probes_zero_is_the_plain_search():
    import torch

    rng = np.random.default_rng(1)
    dim, k = 100, 10
    rows = clustered(rng, 6000, dim)
    orc, ix = pair(zo.L2, dim, rows, 256, 3)
    qs = clustered(rng, 200, dim)
    a = ix.search_batch(qs, k)
    sa = _stats(ix)
    b = ix.search_batch(qs, k, probes=0)
    assert _stats(ix) == sa
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert np.array_equal(a[1], orc.search_batch(qs, k, nthreads=8)[0])
    # the probe entry points themselves at P = 0, host and device
    z = zb()
    o = np.empty((200, k), np.uint64)
    bits = np.empty((200, k), np.uint64)
    c = np.empty(200, np.uint32)
    z._ffi.check(z._ffi.lib().zb_index_search_probe(ix._h, 200, qs.ctypes.data, k, 0, None, o.ctypes.data, bits.ctypes.data,
                                                    c.ctypes.data))
    assert np.array_equal(o, a[1]) and np.array_equal(bits, a[2]) and np.array_equal(c, a[3])
    assert _stats(ix) == sa
    dq = torch.from_numpy(qs).cuda()
    do = torch.empty((200, k), dtype=torch.int64, device="cuda")
    db = torch.empty((200, k), dtype=torch.int64, device="cuda")
    dc = torch.empty(200, dtype=torch.int32, device="cuda")
    z._ffi.check(z._ffi.lib().zb_index_search_probe_device(ix._h, 200, dq.data_ptr(), k, 0, do.data_ptr(), db.data_ptr(),
                                                           dc.data_ptr()))
    torch.cuda.synchronize()
    assert np.array_equal(do.cpu().numpy().view(np.uint64), a[1]) and np.array_equal(dc.cpu().numpy().view(np.uint32), a[3])
    assert _stats(ix) == sa


# ---------------------------------------------------------------- parity sweep
def _sweep_dims(metric):
    return [1, 7, 100, 384, 768, 1040] if metric <= zo.L2 else [7, 100, 768]


@pytest.mark.parametrize("metric", list(METRICS))
@pytest.mark.parametrize("mns", [512, 5])
def test_parity_sweep(metric, mns):
    rng = np.random.default_rng(metric + mns)
    for dim in _sweep_dims(metric):
        n = 3000 if mns > 5 else 1200
        rows = clustered(rng, n, dim)
        orc, ix = pair(metric, dim, rows, mns, 3 if mns > 5 else 6)
        qs = np.concatenate([clustered(rng, 24, dim), rows[:8]])
        for i, k in enumerate(KS):
            parity(orc, ix, qs, k, PS[i % len(PS)], (metric, mns, dim))


def test_cascade_walkers_in_the_tail_kernel():
    # leaves of 32..64 rows, 60 % removed: first leaves often cannot fill k = 16, so the cascade (and, with plan_tail and
    # mns >= 4 k, the tail kernel) runs next to the probe descents
    rng = np.random.default_rng(5)
    dim = 100
    rows = clustered(rng, 4000, dim)
    orc, ix = pair(zo.L2SQ, dim, rows, 64, 4)
    dead = rng.choice(4000, 2400, replace=False)
    orc.remove(dead)
    ix.remove_ordinals(dead.astype(np.uint64))
    qs = clustered(rng, 64, dim)
    for tail in (1, 0):
        ix.set_param("plan_tail", tail)
        for k in (16, 17):
            for p in PS:
                parity(orc, ix, qs, k, p, ("plan_tail", tail))


@pytest.mark.parametrize("metric", [zo.L2, zo.L2SQ, zo.COSINE])
def test_scan_knobs(metric):
    rng = np.random.default_rng(9)
    dim = 768
    rows = clustered(rng, 8000, dim)
    orc, ix = pair(metric, dim, rows, 2047, 3)
    qs = clustered(rng, 64, dim)
    for l2f in (0, 1, 2):
        ix.set_param("l2_filter", l2f)
        for k, p in ((10, 2), (16, 5)):
            parity(orc, ix, qs, k, p, ("l2_filter", l2f))
    ix.set_param("l2_filter", 1)
    ix.set_param("use_tile_scan", 0)
    parity(orc, ix, qs, 10, 5, "use_tile_scan=0")
    assert ix.stats()["last_tile_pairs"] == 0   # no fused kernel: quad_tile / the gather path took every visit
    ix.set_param("use_tile_scan", 1)
    for qt in (0, 1):
        ix.set_param("quad_tile", qt)
        parity(orc, ix, qs, 100, 2, ("quad_tile", qt))


@pytest.mark.parametrize("metric", [zo.L2, zo.COSINE, zo.MANHATTAN])
def test_tombstones_and_incremental_insert(metric):
    rng = np.random.default_rng(11)
    dim = 100
    rows = clustered(rng, 5000, dim)
    orc, ix = pair(metric, dim, rows, 128, 3, load=False)
    qs = clustered(rng, 48, dim)
    for p in (1, 5):
        parity(orc, ix, qs, 10, p, "built")
    dead = rng.choice(5000, 500, replace=False)
    orc.remove(dead)
    ix.remove_ordinals(dead.astype(np.uint64))
    for k, p in ((10, 1), (33, 5), (129, 2)):
        parity(orc, ix, qs, k, p, "tombstones")
    more = clustered(rng, 1500, dim)
    orc.add(more)
    ix.add_raw(more)
    for k, p in ((10, 1), (33, 5), (129, 32)):
        parity(orc, ix, qs, k, p, "insert")


# ---------------------------------------------------------------- ground truth and recall
def _single_plane_forest(rows, trees):
    nodes, coef, cst, leaf_off, members, roots = [], [], [], [0], [], []
    for t in range(trees):
        c, k = zo.make_plane(rows[2 * t], rows[2 * t + 1])
        above = np.array([zo.point_is_above(c, k, x) for x in rows])
        base = len(nodes)
        roots.append(base)
        nodes += [[t, base + 1, base + 2, -1], [-1, -1, -1, 2 * t], [-1, -1, -1, 2 * t + 1]]
        coef.append(c)
        cst.append(k)
        for side in (False, True):
            members += np.flatnonzero(above == side).tolist()
            leaf_off.append(len(members))
    return zo.Forest(nodes, roots, np.stack(coef), cst, leaf_off, members)


@pytest.mark.parametrize("metric", [zo.COSINE, zo.L2SQ, zo.L2])
def test_single_plane_trees_with_a_probe_equal_the_exact_search(metric):
    z = zb()
    rng = np.random.default_rng(13)
    dim, n = 384, 6000
    rows = clustered(rng, n, dim)
    name, _ = METRICS[metric]
    ix = z.LSHIndex(dim, z.LSHIndexOptions(n, 3), getattr(z, name)(), seed=1)
    ix.load_forest(rows, _single_plane_forest(rows, 3))
    ix.remove_ordinals(rng.choice(n, 400, replace=False).astype(np.uint64))
    qs = clustered(rng, 64, dim)
    for k in (1, 10, 100, 128):
        _, o, b, c = ix.search_batch(qs, k, want_ids=False, probes=1)
        _, eo, eb, ec = ix.search_exact_batch(qs, k, want_ids=False)
        assert np.array_equal(c, ec) and np.array_equal(o, eo) and np.array_equal(b, eb), k


def test_recall_never_falls_as_probes_grow():
    z = zb()
    rng = np.random.default_rng(17)
    dim, n, k = 384, 100_000, 10
    c = rng.standard_normal((64, dim)).astype(F32)
    rows = (c[rng.integers(0, 64, n)] + 0.25 * rng.standard_normal((n, dim))).astype(F32)
    qs = (c[rng.integers(0, 64, 1000)] + 0.25 * rng.standard_normal((1000, dim))).astype(F32)
    ix = z.LSHIndex(dim, z.LSHIndexOptions(1024, 2), z.L2Distance(), seed=2)
    ix.add(rows)
    _, eo, _, ec = ix.search_exact_batch(qs, k, want_ids=False)
    truth = [set(eo[i, : ec[i]].tolist()) for i in range(len(qs))]
    prev, recall = None, []
    for p in (0, 1, 2, 4):
        _, o, _, cnt = ix.search_batch(qs, k, want_ids=False, probes=p)
        found = [set(o[i, : cnt[i]].tolist()) & truth[i] for i in range(len(qs))]
        if prev is not None:
            assert all(a <= b for a, b in zip(prev, found)), p
        prev = found
        recall.append(np.mean(z.recall_at_k(o, cnt, eo, ec)))
    assert recall == sorted(recall) and recall[-1] > recall[0], recall


# ---------------------------------------------------------------- stats, entry points, errors
def test_stats_count_the_probe_visits():
    rng = np.random.default_rng(19)
    dim = 64
    rows = clustered(rng, 3000, dim)
    for mns, k in ((5, 10), (256, 10), (64, 33)):
        orc, ix = pair(zo.L2SQ, dim, rows, mns, 4)
        qs = clustered(rng, 40, dim)
        for p in (1, 3, 32):
            parity(orc, ix, qs, k, p)
            expect = sum(int((orc.trace(q, k, probes=p)[:, 3] > 0).sum()) for q in qs)
            assert ix.stats()["last_visits"] == expect, (mns, k, p)
            assert ix.stats()["last_queries"] == len(qs)


def test_entry_points_agree():
    import torch

    z = zb()
    rng = np.random.default_rng(23)
    dim, k, p, nq = 100, 10, 4, 300
    rows = clustered(rng, 8000, dim)
    orc, ix = pair(zo.COSINE, dim, rows, 256, 3)
    qs = clustered(rng, nq, dim)
    parity(orc, ix, qs, k, p)
    ids, o, b, c = ix.search_batch(qs, k, probes=p)
    # device entry point
    dq = torch.from_numpy(qs).cuda()
    do = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    db = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    dc = torch.empty(nq, dtype=torch.int32, device="cuda")
    ix.search_batch_device(nq, dq.data_ptr(), k, do.data_ptr(), db.data_ptr(), dc.data_ptr(), probes=p)
    torch.cuda.synchronize()
    assert np.array_equal(do.cpu().numpy().view(np.uint64), o) and np.array_equal(db.cpu().numpy().view(np.uint64), b)
    assert np.array_equal(dc.cpu().numpy().view(np.uint32), c)
    # slice forms on an unsharded index
    si, so, sb, sc = ix.search_slice(nq, qs, k, probes=p)
    assert np.array_equal(si, ids) and np.array_equal(so, o) and np.array_equal(sb, b) and np.array_equal(sc, c)
    do.zero_()
    ix.search_slice_device(nq, dq.data_ptr(), k, do.data_ptr(), db.data_ptr(), dc.data_ptr(), probes=p)
    torch.cuda.synchronize()
    assert np.array_equal(do.cpu().numpy().view(np.uint64), o)
    # a prefetched call
    po = np.empty((nq, k), np.uint64)
    pb = np.empty((nq, k), np.uint64)
    pc = np.empty(nq, np.uint32)
    ix.search_prefetch_ptr(nq, qs.ctypes.data)
    ix.search_batch_ptr(nq, qs.ctypes.data, k, po.ctypes.data, pb.ctypes.data, pc.ctypes.data, probes=p)
    assert np.array_equal(po, o) and np.array_equal(pb, b) and np.array_equal(pc, c)
    # errors and an index without trees
    with pytest.raises(z._ffi.ZebraError):
        ix.search_batch(qs[:4], k, probes=33)
    ix.search_batch(qs[:4], k, probes=32)
    empty = z.LSHIndex(dim, z.LSHIndexOptions(256, 3), z.CosineDistance(), seed=1)
    _, eo, _, ec = empty.search_batch(qs[:5], k, probes=3)
    assert (ec == 0).all() and (eo == np.uint64(0xFFFFFFFFFFFFFFFF)).all()


def test_database_query_vectors_with_probes():
    z = zb()
    rng = np.random.default_rng(29)
    dim = 64
    rows = clustered(rng, 3000, dim)
    db = z.Database(dim, z.L2SquaredDistance(), index_options=z.LSHIndexOptions(16, 3), seed=4)
    docs = [i.to_bytes(8, "little") for i in range(3000)]
    db.insert_records(rows, docs)
    orc = ProbeOracle(dim, zo.L2SQ, 16, 3, seed=4)
    orc.add(rows)
    qs = clustered(rng, 30, dim)
    res = db.query_vectors(qs, 10, probes=4)
    eo, _, ec = orc.search_batch(qs, 10, nthreads=8, probes=4)
    for q in range(30):
        assert {int.from_bytes(d, "little") for d in res[q].values()} == set(eo[q, : ec[q]].tolist())
    assert db.query_vectors(qs, 10, probes=0) == db.query_vectors(qs, 10)
