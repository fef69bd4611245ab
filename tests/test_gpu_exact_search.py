"""Exact (brute-force) search, zb_index_search_exact*: every result field bit-exact against the oracle's brute force over all
live rows (sorted by (bits, ordinal)), after every mutation path; agreement with the LSH search where both must agree; the
recall helper.  The recall tests at the top are pure numpy."""
import numpy as np
import pytest

from oracle import zb_oracle as zo

F32 = np.float32
SENT = np.uint64(0xFFFFFFFFFFFFFFFF)
METRICS = {zo.COSINE: "CosineDistance", zo.L2SQ: "L2SquaredDistance", zo.L2: "L2Distance"}


def zb():
    import zebra_b200

    return zebra_b200


# ---------------------------------------------------------------- recall_at_k (CPU)
def test_recall_identical_disjoint_and_partial():
    z = zb()
    e = np.array([[1, 2, 3, 4], [5, 6, 7, 8]], np.uint64)
    assert np.array_equal(z.recall_at_k(e, [4, 4], e, [4, 4]), [1.0, 1.0])
    assert np.array_equal(z.recall_at_k(e[::-1].copy(), [4, 4], e, [4, 4]), [0.0, 0.0])
    a = np.array([[4, 3, 9, 10], [8, 0, 0, 0]], np.uint64)
    assert np.allclose(z.recall_at_k(a, [4, 1], e, [4, 4]), [0.5, 0.25])


def test_recall_short_and_empty_lists():
    z = zb()
    e = np.array([[1, 2, SENT], [SENT, SENT, SENT], [3, SENT, SENT]], np.uint64)
    a = np.array([[2, SENT, SENT], [1, 2, 3], [SENT, SENT, SENT]], np.uint64)
    r = z.recall_at_k(a, [1, 3, 0], e, [2, 0, 1])
    assert r.dtype == np.float64 and np.array_equal(r, [0.5, 1.0, 0.0])
    # slots past the counts never count, even when they hold equal values
    assert np.array_equal(z.recall_at_k(e, [0, 0, 0], e, [2, 0, 1]), [0.0, 1.0, 0.0])
    assert z.recall_at_k(np.zeros((0, 3), np.uint64), [], np.zeros((0, 3), np.uint64), []).shape == (0,)


# ---------------------------------------------------------------- helpers (GPU)
def clustered(rng, n, dim, centres=24, noise=0.25):
    c = rng.standard_normal((centres, dim)).astype(F32)
    return (c[rng.integers(0, centres, n)] + noise * rng.standard_normal((n, dim))).astype(F32)


def brute(metric, rows, live, queries, k):
    """(ords [nq,k], bits [nq,k], counts [nq]) of the oracle: live rows by (bits, ordinal)."""
    ords_live = np.flatnonzero(live).astype(np.uint64)
    x = rows[live]
    nq = queries.shape[0]
    o = np.full((nq, k), SENT, np.uint64)
    b = np.full((nq, k), SENT, np.uint64)
    c = np.zeros(nq, np.uint32)
    for q in range(nq):
        if not x.shape[0]:
            continue
        bits = zo.distance_bits_batch(metric, x, np.broadcast_to(queries[q], x.shape))
        top = np.lexsort((ords_live, bits))[:k]
        c[q] = top.size
        o[q, :top.size] = ords_live[top]
        b[q, :top.size] = bits[top]
    return o, b, c


def check(ix, metric, rows, live, queries, k, what=""):
    ids, o, b, c = ix.search_exact_batch(queries, k)
    eo, eb, ec = brute(metric, rows, live, queries, k)
    assert np.array_equal(c, ec), what
    assert np.array_equal(o, eo), what
    assert np.array_equal(b, eb), what
    for q in range(queries.shape[0]):   # ids of the result rows, 0xFF tail
        assert (ids[q, c[q]:] == 0xFF).all(), what
    return ids, o, b, c


def index(z, metric, dim, mns=64, trees=2, seed=3):
    return z.LSHIndex(dim, z.LSHIndexOptions(mns, trees), getattr(z, METRICS[metric])(), seed=seed)


def queries_for(rng, rows, nq):
    nr = min(nq // 2, rows.shape[0])
    return np.concatenate([rows[:nr], clustered(rng, nq - nr, rows.shape[1])]).astype(F32)


# ---------------------------------------------------------------- parity sweep
# (metric, dim, k, rows, queries): dims 1..4672 at the fused kernel's limits, k across the filter (16 / 17), the list width
# (32 / 33) and the longest list, 1 / 15 / 16 / 17 queries, row counts off the range length and below one 64-row stage
SWEEP = [
    (zo.COSINE, 1, 10, 300, 17), (zo.L2SQ, 7, 1, 130, 16), (zo.L2, 100, 16, 5000, 15), (zo.COSINE, 384, 17, 3001, 1),
    (zo.L2SQ, 768, 32, 4100, 16), (zo.L2, 768, 10, 4100, 17), (zo.COSINE, 1024, 33, 2000, 17), (zo.L2SQ, 2240, 100, 1500, 16),
    (zo.L2, 4672, 32, 600, 5), (zo.COSINE, 4384, 128, 600, 5), (zo.L2SQ, 4384, 33, 333, 3), (zo.L2, 384, 128, 200, 16),
    (zo.COSINE, 100, 100, 50, 15), (zo.L2SQ, 16, 10, 63, 17), (zo.L2, 1024, 16, 1000, 16), (zo.L2SQ, 768, 1, 2049, 1),
]


@pytest.mark.gpu
@pytest.mark.parametrize("metric,dim,k,n,nq", SWEEP)
def test_parity_sweep(metric, dim, k, n, nq):
    z = zb()
    rng = np.random.default_rng(dim * 1000 + k)
    rows = clustered(rng, n, dim)
    q = queries_for(rng, rows, nq)
    ix = index(z, metric, dim)
    ix.add(rows)
    live = np.ones(n, bool)
    check(ix, metric, rows, live, q, k)
    dead = rng.choice(n, n // 10, replace=False)
    assert ix.remove_ordinals(dead).all()
    live[dead] = False
    check(ix, metric, rows, live, q, k, "10 % tombstones")


@pytest.mark.gpu
@pytest.mark.parametrize("metric", [zo.COSINE, zo.L2SQ, zo.L2])
def test_fewer_live_rows_than_k(metric):
    z = zb()
    rng = np.random.default_rng(5)
    rows = clustered(rng, 40, 96)
    ix = index(z, metric, 96)
    ix.add(rows)
    live = np.ones(40, bool)
    live[::3] = False
    ix.remove_ordinals(np.flatnonzero(~live))
    _, _, _, c = check(ix, metric, rows, live, queries_for(rng, rows, 9), 100)
    assert (c == live.sum()).all()
    ix.remove_ordinals(np.flatnonzero(live))                          # no live row at all
    _, o, b, c = ix.search_exact_batch(rows[:3], 10)
    assert (c == 0).all() and (o == SENT).all() and (b == SENT).all()


@pytest.mark.gpu
@pytest.mark.parametrize("metric", [zo.COSINE, zo.L2])
def test_multi_chunk_batch(metric):
    """A 1 MiB budget cuts 200 queries over 5000 rows into several chunks; results do not depend on it."""
    z = zb()
    rng = np.random.default_rng(6)
    rows = clustered(rng, 5000, 100)
    q = queries_for(rng, rows, 200)
    ix = index(z, metric, 100)
    ix.add(rows)
    want = ix.search_exact_batch(q, 10)
    ix.set_param("exact_budget_mb", 1)
    got = check(ix, metric, rows, np.ones(5000, bool), q, 10)
    for x, y in zip(want, got):
        assert np.array_equal(x, y)
    with pytest.raises(z.ZebraError):
        ix.set_param("exact_budget_mb", 0)


# ---------------------------------------------------------------- adversarial rows
@pytest.mark.gpu
@pytest.mark.parametrize("metric", [zo.COSINE, zo.L2SQ, zo.L2])
def test_duplicates_straddle_k_and_range_boundaries(metric):
    z = zb()
    rng = np.random.default_rng(7)
    n, dim = 9000, 128
    rows = clustered(rng, n, dim)
    base = rows[17].copy()
    for p in list(range(50, 80)) + list(range(4080, 4110)) + list(range(8180, 8200)):   # across 64-row stages and ranges
        rows[p] = base
    rows[8999] = base
    ix = index(z, metric, dim, mns=512, trees=2)
    ix.add(rows)
    q = np.stack([base, base * F32(2), rows[4100], rows[0]])
    for k in (1, 10, 16, 33, 100):
        _, o, _, _ = check(ix, metric, rows, np.ones(n, bool), q, k, f"k={k}")
    if metric != zo.COSINE:                                          # identical rows: distance 0, ties by ordinal
        assert list(o[0, :5]) == [17, 50, 51, 52, 53]


@pytest.mark.gpu
def test_zero_rows_and_zero_query_cosine():
    z = zb()
    rng = np.random.default_rng(8)
    rows = clustered(rng, 700, 64)
    rows[[3, 64, 65, 400]] = 0
    q = np.concatenate([np.zeros((2, 64), F32), rows[:3], -rows[5:6]])
    ix = index(z, zo.COSINE, 64)
    ix.add(rows)
    for k in (5, 40):
        check(ix, zo.COSINE, rows, np.ones(700, bool), q, k, f"k={k}")


@pytest.mark.gpu
@pytest.mark.parametrize("metric", [zo.L2SQ, zo.L2])
def test_huge_and_non_finite_rows_l2(metric):
    """Rows the dot-product filter cannot bound (huge norms, inf, NaN) are rescanned exactly."""
    z = zb()
    rng = np.random.default_rng(9)
    n, dim = 3000, 256
    rows = clustered(rng, n, dim)
    rows[10] *= F32(1e18)
    rows[11, 3] = np.inf
    rows[12, 7] = np.nan
    rows[2000:2010] *= F32(3e15)
    rows[2500, :] = -np.inf
    # queries: ordinary, near the huge rows, the huge and the inf row themselves, huge norms.  No query holds a NaN: it makes
    # every distance NaN, and a NaN distance carries the device's canonical NaN payload (as in the LSH search), not the host's
    q = np.concatenate([rows[:4], rows[2000:2002] / F32(3e15), rows[10:12], clustered(rng, 3, dim) * F32(1e17)])
    ix = index(z, metric, dim, mns=1024)
    ix.add(rows)
    for k in (1, 10, 16, 17):
        check(ix, metric, rows, np.ones(n, bool), q, k, f"k={k}")


# ---------------------------------------------------------------- every mutation path
@pytest.mark.gpu
@pytest.mark.parametrize("metric", [zo.COSINE, zo.L2])
def test_mutation_paths(metric):
    z = zb()
    rng = np.random.default_rng(10)
    dim, k = 200, 10
    a, b = clustered(rng, 3000, dim), clustered(rng, 700, dim)
    q = queries_for(rng, a, 24)
    ix = index(z, metric, dim)
    ix.add(a)                                                              # bulk
    check(ix, metric, a, np.ones(3000, bool), q, k, "bulk add")
    rows = np.concatenate([a, b])
    ix.add(b[:300])                                                        # incremental, twice
    ix.add(b[300:])
    live = np.ones(3700, bool)
    check(ix, metric, rows, live, np.concatenate([q, b[:5]]), k, "incremental add")
    dead = rng.choice(3700, 400, replace=False)
    ix.remove(ix.export_rows()[1][dead])                                   # remove by id
    live[dead] = False
    check(ix, metric, rows, live, q, k, "remove")
    dup = np.concatenate([rows, rows[:50], rows[100:101]])                 # deduplicate
    ix.add(dup[3700:])
    live = np.concatenate([live, np.ones(51, bool)])
    removed = ix.deduplicate_raw()[1]
    live[removed.astype(np.int64)] = False
    check(ix, metric, dup, live, q, k, "deduplicate")
    ix.clear()                                                             # clear: nothing, then fresh rows
    _, _, _, c = ix.search_exact_batch(q, k)
    assert (c == 0).all()
    ix.add(b)
    check(ix, metric, b, np.ones(700, bool), q, k, "clear + add")
    # load_forest: same row count, different rows -- a cache keyed by the count would return stale norms
    forest = ix.export_forest()
    c2 = (b[::-1] * F32(1.5) + F32(0.25)).astype(F32)
    ix.load_forest(c2, forest)
    check(ix, metric, c2, np.ones(700, bool), q, k, "load_forest")
    T, K = 2, 5                                                            # load_flat
    pick = rng.integers(0, 700, (T * K, 2))
    coef = (c2[pick[:, 1]] - c2[pick[:, 0]]).astype(F32)
    cst = (-(coef * ((c2[pick[:, 0]] + c2[pick[:, 1]]) / F32(2))).sum(1)).astype(F32)
    ix.load_flat(b, K, coef, cst)
    check(ix, metric, b, np.ones(700, bool), q, k, "load_flat")
    blobs, ids = ix.export_tree_blobs(), ix.export_rows()[1]              # import_store: the same store with other values
    perm = rng.permutation(700)
    ix.import_store(ids[perm], c2[perm], blobs)
    got_rows, _, got_live = ix.export_rows()
    assert np.array_equal(got_rows.view(np.uint32), c2.view(np.uint32))   # ordinals follow id order
    check(ix, metric, c2, got_live, q, k, "import_store")


# ---------------------------------------------------------------- entry points and cross-checks
@pytest.mark.gpu
def test_host_and_device_entry_points_agree():
    import torch

    z = zb()
    rng = np.random.default_rng(11)
    rows = clustered(rng, 4000, 100)                                       # 100: padded to 112 on the device
    q = queries_for(rng, rows, 37)
    ix = index(z, zo.L2, 100)
    ix.add(rows)
    ids, o, b, c = ix.search_exact_batch(q, 12)
    _, o2, b2, c2 = ix.search_exact_batch(q, 12, want_ids=False)
    assert np.array_equal(o, o2) and np.array_equal(b, b2) and np.array_equal(c, c2)
    d_q = torch.from_numpy(q).cuda()
    d_o = torch.empty((37, 12), dtype=torch.int64, device="cuda")
    d_b = torch.empty((37, 12), dtype=torch.int64, device="cuda")
    d_c = torch.empty(37, dtype=torch.int32, device="cuda")
    for _ in range(2):
        ix.search_exact_batch_device(37, d_q.data_ptr(), 12, d_o.data_ptr(), d_b.data_ptr(), d_c.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(d_o.cpu().numpy().view(np.uint64), o)
        assert np.array_equal(d_b.cpu().numpy().view(np.uint64), b)
        assert np.array_equal(d_c.cpu().numpy().view(np.uint32), c)
    one = ix.search_exact(q[3], 12)
    assert [bits for _, bits in one] == [int(x) for x in b[3, :c[3]]]
    assert [u.bytes for u, _ in one] == [ids[3, j].tobytes() for j in range(c[3])]


@pytest.mark.gpu
@pytest.mark.parametrize("metric,k", [(zo.COSINE, 10), (zo.L2SQ, 16), (zo.L2, 33), (zo.COSINE, 128)])
def test_one_leaf_per_tree_equals_lsh_search(metric, k):
    """max_node_size above the row count: every tree is one leaf, so the LSH search scores every live row too."""
    z = zb()
    rng = np.random.default_rng(12)
    rows = clustered(rng, 3000, 256)
    ix = index(z, metric, 256, mns=4000, trees=3)
    ix.add(rows)
    ix.remove_ordinals(rng.choice(3000, 200, replace=False))
    q = queries_for(rng, rows, 40)
    _, o, b, c = ix.search_batch(q, k, want_ids=False)
    _, eo, eb, ec = ix.search_exact_batch(q, k, want_ids=False)
    assert np.array_equal(c, ec) and np.array_equal(o, eo) and np.array_equal(b, eb)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["uniform", "clustered"])
def test_invariants_realistic_shape(kind):
    """200k x 768, 4 trees of <= 2048-row leaves: LSH results are live, never beat the exact k-th distance, and carry the
    exact search's bits for every row both return."""
    import torch

    z = zb()
    n, dim, nq, k = 200_000, 768, 512, 10
    d_rows = torch.empty((n, dim), dtype=torch.float32, device="cuda")
    z.synth_fill_device(0, d_rows.data_ptr(), 0, 1, n, dim, 21, 0 if kind == "uniform" else 1)
    ix = z.LSHIndex(dim, z.LSHIndexOptions(2048, 4), z.L2Distance(), seed=21)
    ix.add_device(d_rows.data_ptr(), n)
    dead = np.random.default_rng(13).choice(n, n // 20, replace=False)
    ix.remove_ordinals(dead)
    d_q = torch.empty((nq, dim), dtype=torch.float32, device="cuda")
    z.synth_fill_device(0, d_q.data_ptr(), 0, 1, nq, dim, 22, 0 if kind == "uniform" else 1)
    q = d_q.cpu().numpy()
    _, ao, ab, ac = ix.search_batch(q, k, want_ids=False)
    _, eo, eb, ec = ix.search_exact_batch(q, k, want_ids=False)
    dead_set = set(int(x) for x in dead)
    assert (ec == k).all()
    for i in range(nq):
        assert not dead_set.intersection(int(x) for x in ao[i, :ac[i]])
        if ac[i] == k:
            assert ab[i, k - 1] >= eb[i, k - 1]
        bits_of = dict(zip(eo[i, :ec[i]].tolist(), eb[i, :ec[i]].tolist()))
        for o_, b_ in zip(ao[i, :ac[i]].tolist(), ab[i, :ac[i]].tolist()):
            if o_ in bits_of:
                assert bits_of[o_] == b_
    r = z.recall_at_k(ao, ac, eo, ec)
    assert ((r >= 0) & (r <= 1)).all()
    # a sample against the oracle's brute force over all live rows
    rows = d_rows.cpu().numpy()
    live = np.ones(n, bool)
    live[dead] = False
    so, sb, sc = brute(zo.L2, rows, live, q[:2], k)
    assert np.array_equal(so, eo[:2]) and np.array_equal(sb, eb[:2]) and np.array_equal(sc, ec[:2])


# ---------------------------------------------------------------- errors and statistics
@pytest.mark.gpu
def test_errors_and_stats_untouched():
    z = zb()
    rng = np.random.default_rng(14)
    rows = clustered(rng, 500, 64)
    ix = z.LSHIndex(64, z.LSHIndexOptions(32, 2), z.ManhattanDistance(), seed=1)
    ix.add(rows)
    with pytest.raises(z.ZebraError) as ei:
        ix.search_exact_batch(rows[:2], 10)
    assert ei.value.code == -1
    ix = index(z, zo.L2, 64)
    ix.add(rows)
    with pytest.raises(z.ZebraError) as ei:
        ix.search_exact_batch(rows[:2], 129)
    assert ei.value.code == -1
    _, _, _, c = ix.search_exact_batch(rows[:2], 0)
    assert (c == 0).all()
    for dim, k in ((4688, 10), (4400, 33)):                                # one stage beyond the fused kernel's limit
        big = index(z, zo.COSINE, dim)
        big.add(rng.standard_normal((20, dim)).astype(F32))
        with pytest.raises(z.ZebraError) as ei:
            big.search_exact_batch(rng.standard_normal((1, dim)).astype(F32), k)
        assert ei.value.code == -1
    ix.search_batch(rows[:30], 7)
    before = {k: v for k, v in ix.stats().items() if k.startswith("last_")}
    ix.search_exact_batch(rows[:50], 20)
    after = {k: v for k, v in ix.stats().items() if k.startswith("last_")}
    assert before == after
