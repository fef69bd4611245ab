"""Restricted search on the GPU (zb_index_rowset_*, zb_index_search_*_rowset*, DESIGN 3.10): every result field bit for bit
against the oracle (tests/probe_ref.py's ProbeOracle for P > 0) loaded with the same forest and the complement of the set
removed, across metrics, dims, k, probes, leaf sizes, scan knobs and set sizes; the identities (include-all = plain call,
entry points agree); the lifecycle (remove / add with leaf splits / deduplicate / clear / reload); the exact search on both
sides of the half rule against a brute force; the errors; Database.query_vectors(within=) and the C++ mirror."""
import os
import subprocess
import uuid

import numpy as np
import pytest

from oracle import zb_oracle as zo
from probe_ref import ProbeOracle

pytestmark = pytest.mark.gpu

F32 = np.float32
SENT = np.uint64(0xFFFFFFFFFFFFFFFF)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
METRICS = {zo.COSINE: "CosineDistance", zo.L2SQ: "L2SquaredDistance", zo.L2: "L2Distance", zo.MANHATTAN: "ManhattanDistance",
           zo.HAMMING: "HammingDistance"}


def zb():
    import zebra_b200

    return zebra_b200


def clustered(rng, n, dim, centres=24, noise=0.25):
    c = rng.standard_normal((centres, dim)).astype(F32)
    return (c[rng.integers(0, centres, n)] + noise * rng.standard_normal((n, dim))).astype(F32)


def make(metric, dim, rows, mns, trees, seed=3):
    """(oracle forest, device index loaded with it)."""
    z = zb()
    orc = zo.OracleIndex(dim, metric, mns, trees, seed)
    orc.add(rows)
    forest = orc.export_forest()
    ix = z.LSHIndex(dim, z.LSHIndexOptions(mns, trees), getattr(z, METRICS[metric])(), seed=seed)
    ix.load_forest(rows, forest)
    return forest, ix


def reference(metric, dim, rows, forest, mns, trees, out_rows):
    """The oracle with the same forest and every row of `out_rows` (bool [n]) removed."""
    ref = ProbeOracle(dim, metric, mns, trees)
    ref.load_forest(rows, forest)
    dead = np.flatnonzero(out_rows).astype(np.uint64)
    if dead.size:
        ref.remove(dead)
    return ref


def check(ix, ref, qs, k, probes, rs, what=""):
    ids, o, b, c = ix.search_batch(qs, k, probes=probes, within=rs)
    eo, eb, ec = ref.search_batch(qs, k, nthreads=8, probes=probes)
    assert np.array_equal(c, ec), (what, k, probes)
    assert np.array_equal(o, eo), (what, k, probes)
    assert np.array_equal(b, eb), (what, k, probes)
    for q in range(qs.shape[0]):
        assert (ids[q, c[q]:] == 0xFF).all() and (o[q, c[q]:] == SENT).all()
    return o, b, c


def brute(metric, rows, live, queries, k):
    """Exact top-k over the rows with live[i], by (bits, ordinal)."""
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
        o[q, :top.size], b[q, :top.size] = ords_live[top], bits[top]
    return o, b, c


def sets(rng, n):
    """(name, ordinals, exclude, in-set mask) for the set sizes under test."""
    half = rng.choice(n, n // 2, replace=False)
    one = rng.choice(n, max(1, n // 100), replace=False)
    single = np.array([int(rng.integers(n))])
    out = []
    for name, ords, excl in (("all", np.arange(n), False), ("half", half, False), ("1%", one, False), ("single", single, False),
                             ("empty", np.zeros(0, np.int64), False), ("exclude 1%", one, True)):
        m = np.zeros(n, bool)
        m[ords] = True
        out.append((name, np.concatenate([ords, ords[:3]]), excl, ~m if excl else m))  # a few duplicates in every list
    return out


def _stats(ix):
    return {k: v for k, v in ix.stats().items() if not k.startswith("last_ms") and k != "device_bytes"}


# ---------------------------------------------------------------- parity sweep
KS = [1, 10, 33, 129]
PS = [0, 1, 5]


@pytest.mark.parametrize("metric", list(METRICS))
@pytest.mark.parametrize("mns", [512, 5])
def test_parity_sweep(metric, mns):
    rng = np.random.default_rng(metric * 7 + mns)
    dims = [1, 100, 768, 1040] if metric <= zo.L2 else [1, 100, 768]
    trees = 3 if mns > 5 else 6
    for dim in dims:
        n = 3000 if mns > 5 else 1200
        rows = clustered(rng, n, dim)
        forest, ix = make(metric, dim, rows, mns, trees)
        qs = np.concatenate([clustered(rng, 20, dim), rows[:6]])
        for j, (name, ords, excl, inset) in enumerate(sets(rng, n)):
            with ix.rowset(ordinals=ords, exclude=excl) as rs:
                assert rs.count == int(inset.sum())
                ref = reference(metric, dim, rows, forest, mns, trees, ~inset)
                for i, k in enumerate(KS):
                    check(ix, ref, qs, k, PS[(i + j) % len(PS)], rs, (metric, mns, dim, name))
        ix.close()


@pytest.mark.parametrize("knobs", [{"use_tile_scan": 0}, {"l2_filter": 0}, {"l2_filter": 2}, {"tile_min_rows": 4096}])
def test_scan_knobs(knobs):
    rng = np.random.default_rng(11)
    dim, n, mns, trees = 768, 8000, 2048, 4
    rows = clustered(rng, n, dim)
    forest, ix = make(zo.L2, dim, rows, mns, trees)
    for key, v in knobs.items():
        ix.set_param(key, v)
    qs = np.concatenate([clustered(rng, 40, dim), rows[:8]])
    inset = rng.random(n) < 0.3
    with ix.rowset(ordinals=np.flatnonzero(inset)) as rs:
        ref = reference(zo.L2, dim, rows, forest, mns, trees, ~inset)
        for k, p in ((10, 0), (16, 1), (33, 5)):
            check(ix, ref, qs, k, p, rs, knobs)


# ---------------------------------------------------------------- identities
def test_include_all_equals_the_plain_call_with_its_stats():
    rng = np.random.default_rng(2)
    dim, n = 768, 6000
    rows = clustered(rng, n, dim)
    _, ix = make(zo.L2, dim, rows, 2048, 4)
    ix.remove_ordinals(np.arange(0, n, 9, dtype=np.uint64))
    qs = clustered(rng, 300, dim)
    ix.set_param("l2_filter", 2)   # no adaptive state between the calls compared
    for p in (0, 2):
        plain = ix.search_batch(qs, 10, probes=p)
        sp = _stats(ix)
        for rs in (ix.rowset(ordinals=np.arange(n)), ix.rowset(ordinals=[], exclude=True)):
            got = ix.search_batch(qs, 10, probes=p, within=rs)
            assert _stats(ix) == sp
            for a, b in zip(plain, got):
                assert np.array_equal(a, b)
            rs.close()


def test_entry_points_agree():
    import torch

    z = zb()
    rng = np.random.default_rng(3)
    dim, n, nq, k = 100, 5000, 200, 10
    rows = clustered(rng, n, dim)
    _, ix = make(zo.COSINE, dim, rows, 256, 4)
    rs = ix.rowset(ordinals=rng.choice(n, 1500, replace=False))
    qs = clustered(rng, nq, dim)
    for p in (0, 3):
        ids, o, b, c = ix.search_batch(qs, k, probes=p, within=rs)
        s_ids, so, sb, sc = ix.search_slice(nq, qs, k, probes=p, within=rs)   # unsharded: the slice is the batch
        assert np.array_equal(o, so) and np.array_equal(b, sb) and np.array_equal(c, sc) and np.array_equal(ids, s_ids)
        single = ix.search(qs[5], k, probes=p, within=rs)
        assert [int(x) for _, x in single] == [int(x) for x in b[5, :c[5]]]
        dq = torch.from_numpy(qs).cuda()
        for fn in (ix.search_batch_device, ix.search_slice_device):
            do = torch.empty((nq, k), dtype=torch.int64, device="cuda")
            db = torch.empty((nq, k), dtype=torch.int64, device="cuda")
            dc = torch.empty(nq, dtype=torch.int32, device="cuda")
            fn(nq, dq.data_ptr(), k, do.data_ptr(), db.data_ptr(), dc.data_ptr(), probes=p, within=rs)
            torch.cuda.synchronize()
            assert np.array_equal(do.cpu().numpy().view(np.uint64), o) and np.array_equal(db.cpu().numpy().view(np.uint64), b)
            assert np.array_equal(dc.cpu().numpy().view(np.uint32), c)
    # the device form of the rowset itself
    ords = torch.from_numpy(rng.choice(n, 1500, replace=False).astype(np.int64)).cuda()
    h, cnt = z._ffi.C.c_void_p(), z._ffi.C.c_uint64()
    z._ffi.check(z._ffi.lib().zb_index_rowset_from_ordinals_device(ix._h, 1500, ords.data_ptr(), 0, z._ffi.C.byref(cnt),
                                                                   z._ffi.C.byref(h)))
    rd = z.RowSet(ix, h, int(cnt.value))
    assert rd.count == 1500
    ref = ix.rowset(ordinals=ords.cpu().numpy())
    for a, b_ in zip(ix.search_batch(qs, k, within=rd), ix.search_batch(qs, k, within=ref)):
        assert np.array_equal(a, b_)
    rd.close()
    ref.close()
    rs.close()


# ---------------------------------------------------------------- lifecycle
def test_rowset_follows_remove_add_and_deduplicate():
    rng = np.random.default_rng(4)
    dim, n, mns, trees, k = 64, 3000, 64, 5, 10
    rows = clustered(rng, n, dim)
    z = zb()
    twin = ProbeOracle(dim, zo.L2SQ, mns, trees, seed=3)
    twin.add(rows)
    ix = z.LSHIndex(dim, z.LSHIndexOptions(mns, trees), z.L2SquaredDistance(), seed=3)
    ix.load_forest(rows, twin.export_forest())
    inset = np.zeros(n, bool)
    inset[rng.choice(n, 1200, replace=False)] = True
    rs = ix.rowset(ordinals=np.flatnonzero(inset))
    qs = np.concatenate([clustered(rng, 30, dim), rows[:10]])

    def expect(p):
        allrows = twin.rows
        out = np.ones(allrows.shape[0], bool)
        out[:n] = ~inset
        ref = ProbeOracle(dim, zo.L2SQ, mns, trees)
        ref.load_forest(allrows, twin.export_forest())
        dead = np.flatnonzero(out | twin.tomb).astype(np.uint64)
        ref.remove(dead)
        return ref

    check(ix, expect(0), qs, k, 0, rs, "fresh")
    check(ix, expect(2), qs, k, 2, rs, "fresh")   # derived once; later calls reuse it
    dead = rng.choice(n, 500, replace=False).astype(np.uint64)
    ix.remove_ordinals(dead)
    twin.remove(dead)
    check(ix, expect(0), qs, k, 0, rs, "after remove")
    more = np.concatenate([rows[rng.integers(0, n, 800)] + F32(0.01), clustered(rng, 800, dim)]).astype(F32)
    leaves = ix.stats()["leaves"]
    ix.add(more)
    twin.add(more)
    assert ix.stats()["leaves"] > leaves   # the insert split leaves
    check(ix, expect(0), qs, k, 0, rs, "after add")
    check(ix, expect(1), qs, k, 1, rs, "after add")
    o, _, c = ix.search_batch(np.concatenate([qs, more[:20]]), 33, within=rs)[1:]
    assert (o[o != SENT] < n).all()   # rows added after the rowset never appear
    dup = np.concatenate([rows[np.flatnonzero(inset)[:40]]]).astype(F32)   # copies of rows of the set: deduplicate removes the copies
    ix.add(dup)
    twin.add(dup)
    removed = ix.deduplicate_raw()[1]
    twin.remove(np.sort(removed))
    check(ix, expect(0), qs, k, 0, rs, "after deduplicate")
    # clear / reload reuse ordinals
    ix.load_forest(rows, _forest_of(rows, dim, mns, trees))
    with pytest.raises(z.ZebraError) as e:
        ix.search_batch(qs, k, within=rs)
    assert e.value.code == -5
    rs.close()
    rs = ix.rowset(ordinals=[1, 2, 3])
    ix.clear()
    with pytest.raises(z.ZebraError) as e:
        ix.search_exact_batch(qs, k, within=rs)
    assert e.value.code == -5
    rs.close()
    ix.close()


def _forest_of(rows, dim, mns, trees):
    o = zo.OracleIndex(dim, zo.L2SQ, mns, trees, 3)
    o.add(rows)
    return o.export_forest()


# ---------------------------------------------------------------- exact search
@pytest.mark.parametrize("metric", [zo.COSINE, zo.L2SQ, zo.L2])
def test_exact_both_sides_of_the_half_rule(metric):
    z = zb()
    rng = np.random.default_rng(20 + metric)
    dim, n = 768, 6000
    rows = clustered(rng, n, dim)
    rows[100:140] = rows[3000:3040]   # duplicate rows: ties broken by ordinal
    ix = z.LSHIndex(dim, z.LSHIndexOptions(2048, 2), getattr(z, METRICS[metric])(), seed=1)
    ix.add(rows)
    dead = rng.choice(n, 600, replace=False)
    ix.remove_ordinals(dead.astype(np.uint64))
    live = np.ones(n, bool)
    live[dead] = False
    qs = np.concatenate([clustered(rng, 30, dim), rows[100:110], rows[3000:3005]])
    for frac in (0.05, 0.4, 0.9):   # compacted (<= half of the slots), compacted, masked
        inset = rng.random(n) < frac
        with ix.rowset(ordinals=np.flatnonzero(inset)) as rs:
            for k in (1, 10, 16, 33, 128):
                _, o, b, c = ix.search_exact_batch(qs, k, within=rs)
                eo, eb, ec = brute(metric, rows, live & inset, qs, k)
                assert np.array_equal(c, ec) and np.array_equal(o, eo) and np.array_equal(b, eb), (frac, k)
            # rows of the set removed after the first call (the compacted store refreshes its mask)
            gone = np.flatnonzero(inset & live)[::5]
            ix.remove_ordinals(gone.astype(np.uint64))
            live[gone] = False
            _, o, b, c = ix.search_exact_batch(qs, 10, within=rs)
            eo, eb, ec = brute(metric, rows, live & inset, qs, 10)
            assert np.array_equal(c, ec) and np.array_equal(o, eo) and np.array_equal(b, eb), frac
    ix.close()


def test_exact_device_form_and_stats_untouched():
    import torch

    rng = np.random.default_rng(8)
    dim, n, nq, k = 100, 4000, 50, 10
    rows = clustered(rng, n, dim)
    _, ix = make(zo.L2, dim, rows, 256, 3)
    qs = clustered(rng, nq, dim)
    ix.search_batch(qs, k)
    st = ix.stats()
    with ix.rowset(ordinals=np.arange(0, n, 3)) as rs:
        _, o, b, c = ix.search_exact_batch(qs, k, within=rs)
        assert {a: v for a, v in ix.stats().items() if a != "device_bytes"} == {a: v for a, v in st.items() if a != "device_bytes"}
        dq = torch.from_numpy(qs).cuda()
        do = torch.empty((nq, k), dtype=torch.int64, device="cuda")
        db = torch.empty((nq, k), dtype=torch.int64, device="cuda")
        dc = torch.empty(nq, dtype=torch.int32, device="cuda")
        ix.search_exact_batch_device(nq, dq.data_ptr(), k, do.data_ptr(), db.data_ptr(), dc.data_ptr(), within=rs)
        torch.cuda.synchronize()
        assert np.array_equal(do.cpu().numpy().view(np.uint64), o) and np.array_equal(dc.cpu().numpy().view(np.uint32), c)
        assert np.array_equal(db.cpu().numpy().view(np.uint64), b)
        live = np.zeros(n, bool)
        live[::3] = True
        eo, eb, ec = brute(zo.L2, rows, live, qs, k)
        assert np.array_equal(o, eo) and np.array_equal(b, eb)


# ---------------------------------------------------------------- errors, memory, hosts
def test_errors():
    z = zb()
    rng = np.random.default_rng(9)
    dim, n = 32, 500
    rows = clustered(rng, n, dim)
    _, ix = make(zo.L2, dim, rows, 64, 2)
    _, other = make(zo.L2, dim, rows, 64, 2)
    qs = rows[:4]
    with pytest.raises(z.ZebraError) as e:
        ix.rowset(ordinals=[0, n])
    assert e.value.code == -1
    with pytest.raises(z.ZebraError) as e:   # an undefined flag bit
        z._ffi.check(z._ffi.lib().zb_index_rowset_from_ordinals(ix._h, 1, np.zeros(1, np.uint64).ctypes.data, 2, None,
                                                                z._ffi.C.byref(z._ffi.C.c_void_p())))
    assert e.value.code == -1
    import torch

    bad = torch.tensor([1, n + 5], dtype=torch.int64, device="cuda")
    with pytest.raises(z.ZebraError) as e:
        z._ffi.check(z._ffi.lib().zb_index_rowset_from_ordinals_device(ix._h, 2, bad.data_ptr(), 0, None,
                                                                       z._ffi.C.byref(z._ffi.C.c_void_p())))
    assert e.value.code == -1
    ids = ix.export_rows(0, 3)[1]
    unknown = bytes(16 * [0x42])
    rs = ix.rowset(ids=[bytes(ids[0]), unknown, bytes(ids[2]), bytes(ids[2])])
    assert rs.count == 2 and rs.found.tolist() == [True, False, True, True]
    with pytest.raises(z.ZebraError) as e:
        z._ffi.check(z._ffi.lib().zb_index_search_rowset(other._h, 4, qs.ctypes.data, 5, 0, rs._h, None,
                                                         np.empty(20, np.uint64).ctypes.data, np.empty(20, np.uint64).ctypes.data,
                                                         np.empty(4, np.uint32).ctypes.data))
    assert e.value.code == -1
    with pytest.raises(ValueError):
        other.search_batch(qs, 5, within=rs)
    with pytest.raises(z.ZebraError) as e:
        ix.search_batch(qs, 5, probes=33, within=rs)
    assert e.value.code == -1
    rs.close()
    rs.close()   # idempotent
    # a closed set is refused by every form: the C ABI's NULL rowset would be the unrestricted search
    for call in (lambda: ix.search_batch(qs, 5, within=rs), lambda: ix.search(qs[0], 5, within=rs),
                 lambda: ix.search_slice(4, qs, 5, within=rs), lambda: ix.search_exact_batch(qs, 5, within=rs)):
        with pytest.raises(ValueError):
            call()
    other.close()
    ix.close()


def test_device_bytes_count_the_rowset():
    rng = np.random.default_rng(10)
    dim, n = 128, 20000
    rows = clustered(rng, n, dim)
    _, ix = make(zo.L2, dim, rows, 1024, 2)
    ix.search_batch(rows[:10], 10)
    base = ix.stats()["device_bytes"]
    rs = ix.rowset(ordinals=np.arange(0, n, 50))
    ix.search_exact_batch(rows[:10], 10, within=rs)   # 2 % of the rows: gathered into the rowset's own store
    assert ix.stats()["device_bytes"] >= base + (n // 50) * dim * 4
    rs.close()
    ix.close()


def test_database_query_vectors_within():
    z = zb()
    rng = np.random.default_rng(12)
    dim = 48
    db = z.Database(dim, z.L2Distance(), index_options=z.LSHIndexOptions(64, 4), seed=2)
    rows = clustered(rng, 1500, dim)
    ids = db.insert_records(rows, [b"d%d" % i for i in range(1500)])
    allowed = ids[::4]
    got = db.query_vectors(rows[:20], 5, within=allowed + [uuid.uuid4()])
    with db.index.rowset(ids=allowed) as rs:
        want = db.query_vectors(rows[:20], 5, within=rs)
    assert got == want
    ok = set(allowed)
    assert all(set(v) <= ok for v in got.values())
    assert all(v for v in got.values())   # every query is a row of the index: its leaves hold rows of the set


def test_cpp_mirror(tmp_path):
    zo.build()
    out = str(tmp_path / "rowset_mirror_test")
    lib, orc = os.path.join(ROOT, "zebra_b200"), os.path.join(ROOT, "oracle")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-o", out,
                           os.path.join(ROOT, "tests", "cpp", "rowset_mirror_test.cpp"), f"-L{lib}", "-lzebra_b200", f"-L{orc}",
                           "-lzb_oracle", f"-Wl,-rpath,{lib}", f"-Wl,-rpath,{orc}"])
    r = subprocess.run([out, "gpu"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "all ok" in r.stdout and "MISMATCH" not in r.stdout, r.stdout[-4000:] + r.stderr[-2000:]
