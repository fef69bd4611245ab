"""Rows longer than 768 floats on a GPU.  Above 992 padded dimensions the fused leaf-tile scan no longer fits 16-query tiles
next to its ring: it runs 8-query tiles (1008 .. 2208, n' <= 32), then 4-query tiles (2224 .. 4672), and beyond that the
visits go to quad_tile (up to 3072) or to the per-pair kernels; lists of up to 128 entries switch earlier (8 queries from
720, 4 from 1936, none from 4400).  The dot-product filter for L2 / L2 squared runs inside the fused kernel at every one of
these capacities.  Each case here is checked bit for bit against the CPU oracle (ids, distance bits, counts) and asserts
through stats() which path took it, with the tile capacity derived from the header's own shared-memory layout
(test_scan3.t3_config over t3_layout) and the device's opt-in limit."""
import numpy as np
import pytest

from oracle import zb_oracle as zo
from test_scan3 import build_emu, load_emu, t3_config

pytestmark = pytest.mark.gpu
F32 = np.float32
METRICS = [(zo.COSINE, "CosineDistance"), (zo.L2SQ, "L2SquaredDistance"), (zo.L2, "L2Distance")]
FILTER_MAX_K = 16             # ZB_L2_FILTER_MAX_K: L2 / L2 squared lists the filter takes


def zb():
    import zebra_b200

    return zebra_b200


@pytest.fixture(scope="module")
def layout_lib(tmp_path_factory):
    """The CPU build of zb_scan3_kernel.cuh (tests/scan3_emu.cpp): only its t3_layout is used here."""
    out = str(tmp_path_factory.mktemp("s3") / "libscan3_layout.so")
    build_emu(out)
    return load_emu(out)


def fused_config(lib, dim, k):
    """(qcap, nst) the library picks for this row length and list length, None where the fused kernel does not run."""
    import torch

    if not 1 <= k <= 128:
        return None
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    return t3_config(lib, (dim + 15) // 16 * 16, 1 if k <= 32 else 4, optin)


def clustered(rng, n, dim, centres=32, noise=0.25):
    c = rng.standard_normal((centres, dim)).astype(F32)
    return (c[rng.integers(0, centres, n)] + noise * rng.standard_normal((n, dim))).astype(F32)


def rows_and_queries(rng, n, dim, nq):
    """Clustered rows with a block of exact duplicates and a group of near duplicates (one ulp apart in one coordinate:
    the cancellation the filter's error bound is for); queries: fresh, stored rows, and stored rows lightly perturbed."""
    rows = clustered(rng, n, dim)
    rows[n // 2:n // 2 + 100] = rows[:100]
    for i in range(1, 40):
        rows[200 + i] = rows[200]
        c = i % dim
        rows[200 + i, c] = np.nextafter(rows[200, c], F32(np.inf) if i % 2 else F32(-np.inf), dtype=F32)
    fresh = clustered(rng, nq // 2, dim)
    pick = rows[rng.integers(0, n, nq - nq // 2)].copy()
    pick[::2] += (1e-3 * rng.standard_normal(pick[::2].shape)).astype(F32)
    queries = np.concatenate([fresh, pick]).astype(F32)
    queries[0] = rows[200]
    queries[1] = rows[0]
    return rows, queries


def assert_equal_to(expected, got):
    eo, eb, ec = expected
    _, ords, bits, counts = got
    assert np.array_equal(counts, ec)
    for q in range(ec.size):
        c = int(ec[q])
        assert np.array_equal(ords[q, :c], eo[q, :c]), f"query {q}: ids differ"
        assert np.array_equal(bits[q, :c], eb[q, :c]), f"query {q}: distance bits differ"
        assert np.all(ords[q, c:] == np.iinfo(np.uint64).max)


def assert_path(st, cfg, dim, k, metric, l2_filter):
    """The path stats() reports is the one the shared-memory layout predicts for (dim, k)."""
    if cfg is None:
        assert st["last_tile_pairs"] == 0 and st["last_filter_used"] == 0, (dim, k, st)
        if (dim + 15) // 16 * 16 > 3072:                           # quad_tile does not fit either: per-pair kernels
            assert st["last_tiles"] == 0, (dim, k, st)
        return
    assert st["last_tile_pairs"] > 0.95 * st["last_pairs"], (dim, k, st)
    assert st["last_tiles"] * cfg[0] >= st["last_tile_visits"], (dim, k, cfg, st)   # no tile holds more than qcap queries
    want = int(l2_filter == 2 and metric != zo.COSINE and k <= FILTER_MAX_K and dim >= 128)
    assert st["last_filter_used"] == want, (dim, k, l2_filter, st)


# ------------------------------------------------------------------------------------------ which path runs where
@pytest.mark.parametrize("dim,k", [(992, 10), (1008, 10), (2208, 10), (2224, 10), (4672, 10), (4688, 10),
                                   (704, 100), (720, 100), (1920, 100), (1936, 100), (4384, 100), (4400, 100)])
def test_path_probe_at_the_capacity_boundaries(layout_lib, dim, k):
    """One leaf per tree and exactly 16 queries: every query visits every tree's leaf, so the fused kernel cuts T * 16 / qcap
    tiles -- the tile count tells which capacity ran.  L2 with the filter forced on for n' <= 16."""
    z = zb()
    rng = np.random.default_rng(dim + k)
    n, trees = 700, 3
    rows, queries = rows_and_queries(rng, n, dim, 16)
    orc = zo.OracleIndex(dim, zo.L2, n + 1, trees, seed=4)      # a node splits once it holds max_node_size rows
    orc.add(rows)
    ix = z.LSHIndex(dim, z.LSHIndexOptions(n + 1, trees), z.L2Distance(), seed=4)
    ix.load_forest(rows, orc.export_forest())
    assert ix.stats()["nodes"] == trees
    ix.set_param("l2_filter", 2)
    cfg = fused_config(layout_lib, dim, k)
    for llw in ((8, 4) if k > 32 else (8,)):
        ix.set_param("long_list_warps", llw)
        assert_equal_to(orc.search_batch(queries, k, nthreads=8), ix.search_batch(queries, k, want_ids=False))
        st = ix.stats()
        assert_path(st, cfg, dim, k, zo.L2, 2)
        if cfg is not None:
            assert st["last_tile_visits"] == trees * 16 and st["last_tiles"] == trees * 16 // cfg[0], (dim, k, cfg, st)
        else:
            assert st["last_tiles"] == 0, st
    ix.close()


# ------------------------------------------------------------------------------------------ search parity across the range
K_ALL = (1, 10, 16, 17, 32, 33, 100, 128, 129)


@pytest.mark.parametrize("dim", [1, 7, 1024, 1030, 1536, 2240, 2250, 3072, 3088, 4096, 4688])
@pytest.mark.parametrize("mid,mname", METRICS)
def test_search_parity_across_dims(layout_lib, dim, mid, mname):
    """Device-built forest (leaves up to 2048 rows), every list length class (KR = 1 and 4, past 128: the fused kernel's
    limit), the filter off and forced on, both team shapes for long lists, before and after 10 % tombstones."""
    z = zb()
    rng = np.random.default_rng(dim * 3 + mid)
    n, mns, trees, nq = 12_000, 2048, 3, 200
    rows, queries = rows_and_queries(rng, n, dim, nq)
    orc = zo.OracleIndex(dim, mid, mns, trees, seed=9)
    orc.add(rows)
    ix = z.LSHIndex(dim, z.LSHIndexOptions(mns, trees), getattr(z, mname)(), seed=9)
    ix.add(rows)
    for phase in ("built", "tombstoned"):
        if phase == "tombstoned":
            dead = rng.choice(n, n // 10, replace=False).astype(np.uint64)
            assert np.array_equal(ix.remove_ordinals(dead), orc.remove(dead))
        for k in K_ALL:
            exp = orc.search_batch(queries, k, nthreads=8)
            cfg = fused_config(layout_lib, dim, k)
            filters = (0, 2) if mid != zo.COSINE and k <= FILTER_MAX_K else (1,)
            shapes = (8, 4) if 32 < k <= 128 else (8,)
            for l2f in filters:
                for llw in shapes:
                    ix.set_param("l2_filter", l2f)
                    ix.set_param("long_list_warps", llw)
                    assert_equal_to(exp, ix.search_batch(queries, k, want_ids=False))
                    assert_path(ix.stats(), cfg, dim, k, mid, l2f)
    ix.close()


# ------------------------------------------------------------------------------------------ fallbacks and knobs
def _oracle_and_index(dim, mid, mname, n=8000, mns=2048, trees=3, seed=6, args=()):
    z = zb()
    rng = np.random.default_rng(dim + mid + 17)
    rows, queries = rows_and_queries(rng, n, dim, 150)
    orc = zo.OracleIndex(dim, mid, mns, trees, seed=seed)
    orc.add(rows)
    ix = z.LSHIndex(dim, z.LSHIndexOptions(mns, trees), getattr(z, mname)(*args), seed=seed)
    ix.load_forest(rows, orc.export_forest())
    return orc, ix, queries


@pytest.mark.parametrize("dim", [1024, 2048])
def test_second_generation_scan_and_no_tile_scan(dim):
    """scan_gen = 2 (8-query tiles of the second generation, shared memory up to 1808 floats per row; at 2048 the visits go to
    quad_tile) and use_tile_scan = 0 (no fused kernel at all)."""
    orc, ix, queries = _oracle_and_index(dim, zo.L2SQ, "L2SquaredDistance")
    for k in (10, 32):
        exp = orc.search_batch(queries, k, nthreads=8)
        ix.set_param("scan_gen", 2)
        assert_equal_to(exp, ix.search_batch(queries, k, want_ids=False))
        st = ix.stats()
        assert (st["last_tile_pairs"] > 0) == (dim <= 1808) and st["last_filter_used"] == 0, st
        ix.set_param("scan_gen", 3)
        ix.set_param("use_tile_scan", 0)
        assert_equal_to(exp, ix.search_batch(queries, k, want_ids=False))
        st = ix.stats()
        assert st["last_tile_pairs"] == 0 and st["last_tiles"] > 0, st      # quad_tile took every visit
        ix.set_param("use_tile_scan", 1)
    ix.close()


@pytest.mark.parametrize("dim", [3072, 3088])
@pytest.mark.parametrize("mid,mname", METRICS[::2])
def test_quad_tile_limit(dim, mid, mname):
    """Lists longer than the fused kernel takes (k = 129): quad_tile up to 3072 floats per row, per-pair kernels beyond; and
    with quad_tile off."""
    orc, ix, queries = _oracle_and_index(dim, mid, mname)
    exp = orc.search_batch(queries, 129, nthreads=8)
    for qt in (1, 0):
        ix.set_param("quad_tile", qt)
        assert_equal_to(exp, ix.search_batch(queries, 129, want_ids=False))
        st = ix.stats()
        assert st["last_tile_pairs"] == 0 and (st["last_tiles"] > 0) == (qt == 1 and dim <= 3072), (qt, st)
    ix.close()


@pytest.mark.parametrize("dim", [1536, 3072, 3088])
@pytest.mark.parametrize("mid,mname,args", [(zo.MANHATTAN, "ManhattanDistance", ()), (zo.MINKOWSKI(3), "MinkowskiDistance", (3,))],
                         ids=["Manhattan", "Minkowski3"])
def test_scalar_metrics_seq_tile_limit(dim, mid, mname, args):
    """The sequential-fold tile scan of the scalar metrics fits rows up to 3072 floats; beyond, and with seq_tile = 0, one
    thread folds each pair.  At 1536 floats the tile's queries take exactly the 48 KB a launch gets without opting in."""
    orc, ix, queries = _oracle_and_index(dim, mid, mname, n=5000, args=args)
    for k in (10, 100):
        exp = orc.search_batch(queries, k, nthreads=8)
        for seq in (1, 0):
            ix.set_param("seq_tile", seq)
            assert_equal_to(exp, ix.search_batch(queries, k, want_ids=False))
            assert (ix.stats()["last_tiles"] > 0) == (seq == 1 and dim <= 3072), (k, seq, ix.stats())
    ix.close()


def test_plan_tail_off_and_tile_queries():
    """plan_tail = 0 (one plan-walk kernel) and tile_queries 1, 3, 5, 7 at 1024 dimensions (tiles smaller than the capacity
    of 8 the layout allows there)."""
    orc, ix, queries = _oracle_and_index(1024, zo.L2, "L2Distance")
    exp = orc.search_batch(queries, 10, nthreads=8)
    ix.set_param("plan_tail", 0)
    assert_equal_to(exp, ix.search_batch(queries, 10, want_ids=False))
    ix.set_param("plan_tail", 1)
    for tq in (1, 3, 5, 7):
        ix.set_param("tile_queries", tq)
        assert_equal_to(exp, ix.search_batch(queries, 10, want_ids=False))
        st = ix.stats()
        assert st["last_tile_pairs"] > 0.95 * st["last_pairs"] and st["last_tiles"] * tq >= st["last_tile_visits"], (tq, st)
    ix.close()


# ------------------------------------------------------------------------------------------ device build and hash
@pytest.mark.parametrize("dim", [880, 896, 1584, 1600, 4096])
def test_build_and_hash_variants(dim):
    """Forest arrays of the device build and hash() keys, depths and leaves, bit-exact against the oracle for hash_variant
    0 / 1 / 2 and classify_variant 0 / 1 (rows staged in shared memory up to 1584 and 880 floats respectively, the other
    kernels beyond)."""
    z = zb()
    rng = np.random.default_rng(dim)
    n, mns, trees = 3000, 64, 3
    rows = clustered(rng, n, dim)
    rows[1500:1520] = rows[:20]
    orc = zo.OracleIndex(dim, zo.L2SQ, mns, trees, seed=13)
    orc.add(rows)
    fa = orc.export_forest()
    probe = np.concatenate([rows[:300], clustered(rng, 200, dim)]).astype(F32)
    ek, ed, el = orc.hash(probe)
    for hv in (0, 1, 2):
        for cv in (0, 1):
            ix = z.LSHIndex(dim, z.LSHIndexOptions(mns, trees), z.L2SquaredDistance(), seed=13)
            ix.set_param("hash_variant", hv)
            ix.set_param("classify_variant", cv)
            ix.add(rows)
            fb = ix.export_forest()
            for name in ("roots", "nodes", "cst", "coef", "leaf_off", "members"):
                assert np.array_equal(getattr(fa, name), getattr(fb, name)), (hv, cv, name)
            keys, depth, leaf = ix.hash(probe)
            assert np.array_equal(keys, ek) and np.array_equal(depth, ed) and np.array_equal(leaf, el), (hv, cv)
            ix.close()
