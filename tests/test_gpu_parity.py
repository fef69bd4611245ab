"""Parity tests proper: the CUDA path (through the C ABI of libzebra_b200.so) against the CPU oracle on the same
seeded inputs.  Bar: bucket keys, ids/ordinals and counts bit-exact (ties by id); distance bits bit-exact against
the oracle (which itself is within 1e-5 relative of simsimd's approximate-rsqrt cosine, see oracle header)."""
import struct
import uuid

import numpy as np
import pytest

from oracle import zb_oracle as zo

pytestmark = pytest.mark.gpu

METRICS = [(zo.COSINE, "CosineDistance"), (zo.L2SQ, "L2SquaredDistance"), (zo.L2, "L2Distance")]


def zb():
    import zebra_b200

    return zebra_b200


def metric_obj(name):
    return getattr(zb(), name)()


def f64bits(x):
    return struct.unpack("<Q", struct.pack("<d", float(x)))[0]


def clustered(rng, n, dim, centres=32, noise=0.25):
    c = rng.standard_normal((centres, dim)).astype(np.float32)
    return (c[rng.integers(0, centres, n)] + noise * rng.standard_normal((n, dim))).astype(np.float32)


def make_queries(rng, rows, nq):
    """half fresh draws, half stored rows (exact duplicates and lightly perturbed) -- SURVEY 8d."""
    dim = rows.shape[1]
    fresh = rng.standard_normal((nq // 2, dim)).astype(np.float32)
    pick = rows[rng.integers(0, rows.shape[0], nq - nq // 2)].copy()
    pick[::2] += (1e-3 * rng.standard_normal(pick[::2].shape)).astype(np.float32)
    return np.concatenate([fresh, pick]).astype(np.float32)


def assert_search_equal(ix, orc, queries, k, nthreads=8):
    _, ords, bits, counts = ix.search_batch(queries, k, want_ids=False)
    eo, eb, ec = orc.search_batch(queries, k, nthreads=nthreads)
    assert np.array_equal(counts, ec)
    for q in range(queries.shape[0]):
        c = int(ec[q])
        assert np.array_equal(ords[q, :c], eo[q, :c]), f"query {q}: ids differ"
        assert np.array_equal(bits[q, :c], eb[q, :c]), f"query {q}: distance bits differ"
        assert np.all(ords[q, c:] == np.iinfo(np.uint64).max)


# ------------------------------------------------------------------------------------------ arithmetic
@pytest.mark.parametrize("dim", [4, 16, 20, 384, 768, 1024, 4096, 8192])
@pytest.mark.parametrize("mid,mname", METRICS)
def test_metric_bits_exact(dim, mid, mname):
    rng = np.random.default_rng(dim + mid)
    a = rng.standard_normal((513, dim)).astype(np.float32)
    b = rng.standard_normal((513, dim)).astype(np.float32)
    a[0] = 0; b[0] = 0            # both zero
    a[1] = 0                      # one zero
    b[2] = a[2]                   # identical
    b[3] = -a[3]                  # opposite
    a[4] *= 1e-20; b[4] *= 1e-20  # underflowing squares
    a[5] *= 1e18; b[5] *= 1e18    # overflowing squares -> inf
    got = metric_obj(mname).distance_batch(a, b)
    exp = zo.distance_bits_batch(mid, a, b)
    assert np.array_equal(got, exp)
    assert metric_obj(mname).distance(a[7], b[7]) == int(exp[7])


@pytest.mark.parametrize("dim", [16, 40, 384, 768, 1024, 4096, 8192])
def test_point_is_above_bit_exact_including_adversarial(dim):
    rng = np.random.default_rng(dim)
    n = 4096
    coef = rng.standard_normal((n, dim)).astype(np.float32)
    x = rng.standard_normal((n, dim)).astype(np.float32)
    cst = rng.standard_normal(n).astype(np.float32)
    # adversarial: constants within a few ulps of -dot, so dot + c straddles zero
    dots = np.array([np.float32(zo.dot(coef[i], x[i])) for i in range(n)], dtype=np.float32)
    for j, ulps in enumerate((0, 1, -1, 2, -2)):
        sel = slice(j, n // 2, 5)
        v = -dots[sel]
        step = np.nextafter(v, np.float32(np.inf) if ulps > 0 else np.float32(-np.inf)) - v
        cst[sel] = v + abs(ulps) * step if ulps else v
    coef[n - 1] = 0; cst[n - 1] = -0.0                 # +0 + -0 = +0 >= 0 -> above
    coef[n - 2] = 0; cst[n - 2] = -1e-45               # smallest negative subnormal -> below
    coef[n - 3, 0] = np.nan                            # NaN -> below
    got = zb().point_is_above(coef, cst, x)
    exp = zo.above_batch(coef, cst, x).astype(bool)
    assert np.array_equal(got, exp)
    assert got[n - 1] and not got[n - 2] and not got[n - 3]
    assert 0.2 < exp[: n // 2].mean() < 0.9            # the adversarial half really straddles zero


# ------------------------------------------------------------------------------------------ hand-built forest
def test_kat_forest_cascade_truncation_tombstones():
    from test_oracle_walk import kat_forest

    z = zb()
    forest, rows = kat_forest()
    ix = z.LSHIndex(4, z.LSHIndexOptions(max_node_size=6, num_trees=1), z.L2SquaredDistance())
    ix.load_forest(rows, forest)
    q = np.array([-1, -1, 0, 0], dtype=np.float32)
    _, ords, bits, counts = ix.search_batch(q[None], 4)
    assert counts[0] == 4 and ords[0].tolist() == [4, 0, 1, 2]       # Q1 cascade + Q2 truncation (row 5 cut)
    assert bits[0].tolist() == [f64bits(2.25), f64bits(32.0), f64bits(52.0), f64bits(74.0)]
    _, ords, _, counts = ix.search_batch(np.array([[4, 4, 0, 0]], np.float32), 4)
    assert ords[0].tolist() == [6, 7, 8, 9]
    assert ix.remove_ordinals([0]).tolist() == [True]
    assert ix.remove_ordinals([0, 99]).tolist() == [False, False]
    _, ords, _, counts = ix.search_batch(q[None], 4)
    assert ords[0].tolist() == [4, 1, 2, 3]                          # emptied main leaf -> backup gets n = 4
    _, ords, bits, counts = ix.search_batch(q[None], 50)             # top_k > live rows -> short result
    assert counts[0] == 10 and sorted(ords[0, :10].tolist()) == list(range(1, 11))
    assert np.all(ords[0, 10:] == np.iinfo(np.uint64).max)
    st = ix.stats()
    assert st["rows"] == 11 and st["live_rows"] == 10


# ------------------------------------------------------------------------------------------ config 1
@pytest.mark.parametrize("mid,mname", METRICS)
def test_config1_defaults_10k_x384_search_parity_on_oracle_forest(mid, mname):
    """BASELINE config 1: 10k x 384, reference defaults (leaf 5, 15 trees), 1k top-10 queries."""
    z = zb()
    rng = np.random.default_rng(100 + mid)
    n, dim, nq, k = 10_000, 384, 1000, 10
    rows = clustered(rng, n, dim)
    orc = zo.OracleIndex(dim, mid, 5, 15, seed=11)
    orc.add(rows)
    forest = orc.export_forest()
    ix = z.LSHIndex(dim, z.LSHIndexOptions(5, 15), metric_obj(mname), seed=11)
    ix.load_forest(rows, forest)
    queries = make_queries(rng, rows, nq)
    assert_search_equal(ix, orc, queries, k)
    # bucket keys of stored rows and of queries
    keys, depth, leaf = ix.hash(queries[:200])
    ek, ed, el = orc.hash(queries[:200])
    assert np.array_equal(keys, ek) and np.array_equal(depth, ed) and np.array_equal(leaf, el)
    # delete 10 % and query again (tombstones)
    dead = rng.choice(n, n // 10, replace=False).astype(np.uint64)
    assert ix.remove_ordinals(dead).all()
    orc.remove(dead)
    assert_search_equal(ix, orc, queries[:300], k)
    _, ords, _, _ = ix.search_batch(queries[:300], k, want_ids=False)
    assert not np.isin(ords, dead).any()


# ------------------------------------------------------------------------------------------ build parity
@pytest.mark.parametrize("n,dim,mns,trees", [(3000, 384, 5, 15), (5000, 768, 64, 4), (2000, 20, 8, 3), (700, 16, 1000, 2)])
def test_device_build_equals_oracle_build(n, dim, mns, trees):
    z = zb()
    rng = np.random.default_rng(n + mns)
    rows = clustered(rng, n, dim)
    orc = zo.OracleIndex(dim, zo.L2SQ, mns, trees, seed=77)
    orc.add(rows)
    ix = z.LSHIndex(dim, z.LSHIndexOptions(mns, trees), z.L2SquaredDistance(), seed=77)
    _, ordinals = ix.add_raw(rows)
    assert ordinals.tolist() == list(range(n))
    fa, fb = orc.export_forest(), ix.export_forest()
    for name in ("roots", "nodes", "cst", "coef", "leaf_off", "members"):
        assert np.array_equal(getattr(fa, name), getattr(fb, name)), name
    assert not ix.no_trees() and not ix.no_vectors() and not ix.is_empty()
    keys, depth, leaf = ix.hash(rows[:500])
    ek, ed, el = orc.hash(rows[:500])
    assert np.array_equal(keys, ek) and np.array_equal(depth, ed) and np.array_equal(leaf, el)
    queries = make_queries(rng, rows, 200)
    assert_search_equal(ix, orc, queries, 10)


def test_duplicate_rows_build_terminates_and_ties_break_by_id():
    z = zb()
    dim = 32
    base = np.random.default_rng(5).standard_normal((40, dim)).astype(np.float32)
    rows = np.repeat(base, 8, axis=0)                     # every row 8 times: forced leaves, many exact ties
    orc = zo.OracleIndex(dim, zo.L2SQ, 4, 3, seed=1)
    orc.add(rows)
    ix = z.LSHIndex(dim, z.LSHIndexOptions(4, 3), z.L2SquaredDistance(), seed=1)
    ix.add(rows)
    fa, fb = orc.export_forest(), ix.export_forest()
    for name in ("roots", "nodes", "cst", "coef", "leaf_off", "members"):
        assert np.array_equal(getattr(fa, name), getattr(fb, name)), name
    assert_search_equal(ix, orc, base[:20], 5)
    _, ords, bits, _ = ix.search_batch(base[:1], 5)
    assert ords[0].tolist() == [0, 1, 2, 3, 4] and bits[0].tolist() == [0] * 5


# ------------------------------------------------------------------------------------------ CRUD
@pytest.mark.parametrize("mid,mname", METRICS[:2])
def test_incremental_add_remove_parity(mid, mname):
    z = zb()
    rng = np.random.default_rng(9 + mid)
    dim, mns, trees = 64, 16, 5
    rows = clustered(rng, 4000, dim)
    orc = zo.OracleIndex(dim, mid, mns, trees, seed=3)
    ix = z.LSHIndex(dim, z.LSHIndexOptions(mns, trees), metric_obj(mname), seed=3)
    queries = make_queries(rng, rows, 120)
    lo = 0
    for step, hi in enumerate((1500, 1501, 2600, 4000)):
        orc.add(rows[lo:hi])
        _, ordinals = ix.add_raw(rows[lo:hi])
        assert ordinals.tolist() == list(range(lo, hi))
        lo = hi
        fa, fb = orc.export_forest(), ix.export_forest()
        for name in ("roots", "nodes", "cst", "coef"):
            assert np.array_equal(getattr(fa, name), getattr(fb, name)), (step, name)
        for l in range(fa.leaf_off.size - 1):   # member ORDER inside a leaf is storage detail; sets must agree
            assert sorted(fa.members[fa.leaf_off[l]:fa.leaf_off[l + 1]]) == sorted(fb.members[fb.leaf_off[l]:fb.leaf_off[l + 1]])
        assert_search_equal(ix, orc, queries, 10)
        dead = rng.choice(hi, 100, replace=False).astype(np.uint64)
        assert np.array_equal(ix.remove_ordinals(dead), orc.remove(dead))
        assert_search_equal(ix, orc, queries, 10)
    assert ix.stats()["live_rows"] == orc.num_live


@pytest.mark.parametrize("k", [1, 3, 10, 100, 700])
def test_topk_range_and_large_leaves(k):
    z = zb()
    rng = np.random.default_rng(k)
    dim, n = 128, 6000
    rows = clustered(rng, n, dim, centres=8)
    orc = zo.OracleIndex(dim, zo.COSINE, 512, 4, seed=2)
    orc.add(rows)
    ix = z.LSHIndex(dim, z.LSHIndexOptions(512, 4), z.CosineDistance(), seed=2)
    ix.add(rows)
    queries = make_queries(rng, rows, 64)
    assert_search_equal(ix, orc, queries, k)
    ix.set_param("use_tile_scan", 0)            # the generic path alone must give the same answer
    assert_search_equal(ix, orc, queries, k)


def test_visit_plan_grows_and_replans():
    """Default forest shape (leaf capacity 5, 15 trees): the count cascade (Q1) makes walkers visit many leaves; starting
    from a 2-slot plan region forces the grow-and-replan loop several times and must not change the answer."""
    z = zb()
    rng = np.random.default_rng(11)
    rows = clustered(rng, 4000, 64)
    orc = zo.OracleIndex(64, zo.L2SQ, 5, 15, seed=4)
    orc.add(rows)
    ix = z.LSHIndex(64, z.LSHIndexOptions(5, 15), z.L2SquaredDistance(), seed=4)
    ix.add(rows)
    ix.set_param("visit_slots", 2)
    assert_search_equal(ix, orc, make_queries(rng, rows, 200), 25)


@pytest.mark.parametrize("mns,trees", [(5, 15), (128, 3)])
def test_deduplicate_matches_oracle(mns, trees):
    """lsh.rs:270-288: the first row (in id order) of every distinct bit pattern stays; +0.0 / -0.0 are different bits."""
    z = zb()
    rng = np.random.default_rng(mns)
    dim, n = 40, 3000
    rows = clustered(rng, n, dim)
    src = rng.integers(0, 200, 600)
    dst = rng.choice(np.arange(200, n), 600, replace=False)
    rows[dst] = rows[src]                                   # 600 copies of 200 originals (chains of duplicates)
    rows[2500] = 0.0; rows[2501] = 0.0; rows[2502] = -0.0   # 2501 duplicates 2500; 2502 has different bits
    orc = zo.OracleIndex(dim, zo.L2SQ, mns, trees, seed=3)
    orc.add(rows)
    ix = z.LSHIndex(dim, z.LSHIndexOptions(mns, trees), z.L2SquaredDistance(), seed=3)
    ix.add(rows)
    pre = np.arange(5, n, 97, dtype=np.uint64)              # rows already removed are neither kept nor counted
    orc.remove(pre); ix.remove_ordinals(pre)
    exp = orc.deduplicate()
    _, got = ix.deduplicate_raw()
    assert np.array_equal(got, exp) and 2501 in got and 2502 not in got
    assert ix.stats()["live_rows"] == orc.num_live
    queries = make_queries(rng, rows, 100)
    assert_search_equal(ix, orc, queries, 10)               # tombstones and live leaf counts followed
    assert ix.deduplicate_raw()[1].size == 0                # idempotent


def test_deduplicate_with_caller_ids_keeps_smallest_id():
    z = zb()
    dim = 16
    base = np.random.default_rng(1).standard_normal((3, dim)).astype(np.float32)
    rows = np.stack([base[0], base[1], base[0], base[2], base[1]])
    ids = [uuid.UUID(int=v) for v in (50, 40, 10, 30, 20)]  # duplicates of row 0: ids 50 and 10 -> 10 stays
    ix = z.LSHIndex(dim, z.LSHIndexOptions(5, 2), z.CosineDistance(), seed=1)
    ix.add(rows, ids)
    removed = ix.deduplicate()
    assert removed == {uuid.UUID(int=50), uuid.UUID(int=40)}


def test_empty_index_and_clear():
    z = zb()
    ix = z.LSHIndex(48, z.LSHIndexOptions(5, 3), z.L2Distance())
    assert ix.no_vectors() and ix.no_trees() and ix.is_empty()
    q = np.zeros((3, 48), np.float32)
    _, ords, bits, counts = ix.search_batch(q, 5)
    assert counts.tolist() == [0, 0, 0] and np.all(ords == np.iinfo(np.uint64).max)
    assert ix.search(q[0], 5) == []
    with pytest.raises(z.ZebraError):
        ix.hash(q)
    rows = np.random.default_rng(0).standard_normal((100, 48)).astype(np.float32)
    ix.add(rows)
    assert not ix.is_empty()
    ix.clear()
    assert ix.is_empty()
    _, ordinals = ix.add_raw(rows[:10])
    assert ordinals.tolist() == list(range(10))


def test_uuid_api_and_database_facade():
    z = zb()
    rng = np.random.default_rng(21)
    dim = 384
    rows = clustered(rng, 2000, dim)
    db = z.Database(dim, z.L2SquaredDistance(), index_options=z.LSHIndexOptions(5, 15), seed=4)
    assert db.query_vectors(rows[:2], 3) == {}
    docs = [i.to_bytes(8, "little") for i in range(2000)]
    ids = db.insert_records(rows, docs)
    assert len(set(ids)) == 2000 and all(i.version == 7 for i in ids[:10])
    assert ids == sorted(ids)                                   # minted ids sort like ordinals (tie-break by id)
    orc = zo.OracleIndex(dim, zo.L2SQ, 5, 15, seed=4)
    orc.add(rows)
    res = db.query_vectors(rows[:50], 10)
    for q in range(50):
        eo, _ = orc.search(rows[q], 10)
        assert {int.from_bytes(d, "little") for d in res[q].values()} == set(eo.tolist())
        assert ids[q] in res[q]
    hit = db.index.search(rows[7], 3, z.L2SquaredDistance())
    assert hit[0] == (ids[7], 0)
    with pytest.raises(ValueError):
        db.index.search(rows[7], 3, z.CosineDistance())
    db.remove([ids[7], uuid.uuid4()])
    assert ids[7] not in db.query_vectors(rows[7:8], 10)[0]
    # caller-supplied ids
    ix = z.LSHIndex(dim, z.LSHIndexOptions(5, 3), z.L2Distance())   # (cosine under Q4 ranks an identical row LATE)
    mine = [uuid.UUID(int=1000 + i) for i in range(100)]
    assert ix.add(rows[:100], ids=mine) == mine
    assert ix.search(rows[5], 1)[0][0] == mine[5]
    assert ix.remove([mine[5]]) == {mine[5]}
    assert ix.search(rows[5], 1)[0][0] != mine[5]


def test_synth_is_deterministic_and_shard_consistent():
    import torch

    z = zb()
    a = torch.empty((1000, 384), dtype=torch.float32, device="cuda")
    b = torch.empty((500, 384), dtype=torch.float32, device="cuda")
    z.synth_fill_device(0, a.data_ptr(), 0, 1, 1000, 384, 5, 1)
    z.synth_fill_device(0, b.data_ptr(), 1, 2, 500, 384, 5, 1)     # rows 1,3,5,... as a 2-way shard would
    torch.cuda.synchronize()
    assert torch.equal(a[1::2], b)
    assert float(a.abs().max()) <= 1.25 and float(a.std()) > 0.3


# ------------------------------------------------------------------------------------------ multi-GPU (NCCL)
def test_sharded_two_gpus_equals_oracle():
    """Bucket-sharded index over 2 GPUs of this box (leaf l on rank l % 2; NCCL: allreduce of leaf counts, send/recv of the
    rows of each leaf to its owner, allgather of the visit plan, all-to-all + allgather of the per-query top-k) against the
    unsharded oracle: bulk build, deletes, incremental insert; shapes of BASELINE configs 1, 2, 3 and 5.  Skipped on a
    single-GPU box."""
    import os
    import subprocess
    import sys

    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29517", os.path.join(root, "tests", "mgpu_parity.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert out.stdout.count(": ok") == 20 and "MISMATCH" not in out.stdout


# ------------------------------------------------------------------------------------------ double-buffered uploads
@pytest.mark.parametrize("dim", [100, 384])
def test_prefetched_batches_give_the_same_answers(dim):
    """zb_index_search_prefetch only moves the upload of an announced batch ahead of the search call that consumes it:
    announced, unannounced, stale and twice-announced batches all return what the oracle returns (lsh.rs:544-565)."""
    rng = np.random.default_rng(77 + dim)
    rows = clustered(rng, 6000, dim)
    ix = zb().LSHIndex(dim, zb().LSHIndexOptions(256, 3), metric_obj("L2Distance"), seed=5)
    orc = zo.OracleIndex(dim, zo.L2, 256, 3, seed=5)
    ix.add(rows); orc.add(rows)
    batches = [np.ascontiguousarray(make_queries(rng, rows, 96 + 8 * i)) for i in range(4)]
    ix.search_prefetch_ptr(batches[0].shape[0], batches[0].ctypes.data)
    for i, q in enumerate(batches):
        if i + 1 < len(batches):                       # announce the next batch, then consume this one
            nxt = batches[i + 1]
            ix.search_prefetch_ptr(nxt.shape[0], nxt.ctypes.data)
        assert_search_equal(ix, orc, q, 10)
    # an announcement nobody consumes, a third one that displaces the oldest, and a search of something else entirely
    ix.search_prefetch_ptr(batches[0].shape[0], batches[0].ctypes.data)
    ix.search_prefetch_ptr(batches[1].shape[0], batches[1].ctypes.data)
    ix.search_prefetch_ptr(batches[2].shape[0], batches[2].ctypes.data)
    other = np.ascontiguousarray(make_queries(rng, rows, 50))
    assert_search_equal(ix, orc, other, 10)
    assert_search_equal(ix, orc, batches[2], 10)
    assert_search_equal(ix, orc, batches[1], 10)
    # fewer rows announced than searched: the call uploads by itself
    ix.search_prefetch_ptr(10, batches[3].ctypes.data)
    assert_search_equal(ix, orc, batches[3], 10)
    ix.close()
