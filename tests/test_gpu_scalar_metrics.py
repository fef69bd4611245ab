"""GPU parity of the ten scalar metrics (distance.rs:51-190, SURVEY 8f row 3): Metric::distance for independent pairs and
LSHIndex::search with each metric, through the C ABI, against the CPU oracle.  Bar: distance bits, ids and counts
bit-exact (the metrics are sequential f32 folds; the device keeps the order, see zebra_b200/csrc/zb_metrics.cuh)."""
import numpy as np
import pytest

from oracle import zb_oracle as zo
from test_scalar_metrics import adversarial

pytestmark = pytest.mark.gpu

SCALAR = [
    (zo.CHEBYSHEV, "ChebyshevDistance", ()), (zo.CANBERRA, "CanberraDistance", ()),
    (zo.BRAY_CURTIS, "BrayCurtisDistance", ()), (zo.MANHATTAN, "ManhattanDistance", ()), (zo.L3, "L3Distance", ()),
    (zo.L4, "L4Distance", ()), (zo.HAMMING, "HammingDistance", ()), (zo.MINKOWSKI(0), "MinkowskiDistance", (0,)),
    (zo.MINKOWSKI(3), "MinkowskiDistance", (3,)), (zo.MINKOWSKI(7), "MinkowskiDistance", (7,)),
    (zo.PNORM(0), "PNormDistance", (0,)), (zo.PNORM(2), "PNormDistance", (2,)), (zo.PNORM(5), "PNormDistance", (5,)),
]
IDS = [f"{n}{a[0] if a else ''}" for _, n, a in SCALAR]


def zb():
    import zebra_b200

    return zebra_b200


def metric_obj(name, args):
    return getattr(zb(), name)(*args)


def clustered(rng, n, dim, centres=32, noise=0.25):
    c = rng.standard_normal((centres, dim)).astype(np.float32)
    return (c[rng.integers(0, centres, n)] + noise * rng.standard_normal((n, dim))).astype(np.float32)


def assert_search_equal(ix, orc, queries, k, nthreads=8):
    _, ords, bits, counts = ix.search_batch(queries, k, want_ids=False)
    eo, eb, ec = orc.search_batch(queries, k, nthreads=nthreads)
    assert np.array_equal(counts, ec)
    for q in range(queries.shape[0]):
        c = int(ec[q])
        assert np.array_equal(ords[q, :c], eo[q, :c]), f"query {q}: ids differ"
        assert np.array_equal(bits[q, :c], eb[q, :c]), f"query {q}: distance bits differ"
        assert np.all(ords[q, c:] == np.iinfo(np.uint64).max)


@pytest.mark.parametrize("dim", [1, 3, 4, 5, 16, 20, 384, 768, 1024, 4096, 8192])
def test_scalar_metric_bits_exact(dim):
    rng = np.random.default_rng(50 + dim)
    a, b = adversarial(rng, 700, dim)
    a[20:60] = np.round(a[20:60] * 4) / 4
    b[20:60] = np.round(b[20:60] * 4) / 4
    for code, name, args in SCALAR:
        m = metric_obj(name, args)
        got = m.distance_batch(a, b)
        exp = zo.distance_bits_batch(code, a, b)
        assert np.array_equal(got, exp), (name, args, dim, np.nonzero(got != exp)[0][:5])
        assert m.distance(a[12], b[12]) == int(exp[12])


def test_minkowski_power_64_and_value_decoding():
    z = zb()
    rng = np.random.default_rng(2)
    a = rng.standard_normal((64, 48)).astype(np.float32)
    b = rng.standard_normal((64, 48)).astype(np.float32)
    m = z.MinkowskiDistance(64)
    got = m.distance_batch(a, b)                                   # |d|^64 overflows f32 for |d| > 4: +inf, as the reference
    assert np.array_equal(got, zo.distance_bits_batch(zo.MINKOWSKI(64), a, b))
    a *= np.float32(0.2); b *= np.float32(0.2)                     # no overflow: the 64-norm is within 48^(1/64) of the max norm
    got = m.distance_batch(a, b)
    assert np.array_equal(got, zo.distance_bits_batch(zo.MINKOWSKI(64), a, b))
    cheb = z.ChebyshevDistance().to_float(z.ChebyshevDistance().distance_batch(a, b))
    val = m.to_float(got)
    assert np.all(val >= cheb * 0.9999) and np.all(val <= cheb * 1.07)
    man = z.ManhattanDistance()
    assert np.allclose(man.to_float(man.distance_batch(a, b)), np.abs(a - b).sum(1), rtol=1e-5)
    ham = z.HammingDistance()
    assert ham.to_float(ham.distance_batch(a, a)).tolist() == [0.0] * 64
    with pytest.raises(ValueError):
        z.MinkowskiDistance(65)


@pytest.mark.parametrize("code,name,args", SCALAR, ids=IDS)
def test_search_parity_default_forest(code, name, args):
    """Reference defaults (leaf capacity 5, 15 trees): the plan, the gather scoring, Q2 truncation and the merge with a
    scalar metric's u64 keys (f32 bits zero-extended)."""
    z = zb()
    rng = np.random.default_rng(300 + (code & 0xFF) + (code >> 8))
    n, dim, nq, k = 3000, 100, 200, 10          # dim % 16 != 0: the fold must stop at dim, not at the padded pitch
    rows = clustered(rng, n, dim)
    rows[5] = 0.0                                # Canberra / Bray-Curtis meet 0/0 when a query is zero too
    orc = zo.OracleIndex(dim, code, 5, 15, seed=21)
    orc.add(rows)
    ix = z.LSHIndex(dim, z.LSHIndexOptions(5, 15), metric_obj(name, args), seed=21)
    ix.add(rows)
    fa, fb = orc.export_forest(), ix.export_forest()
    for f in ("roots", "nodes", "cst", "coef", "leaf_off", "members"):
        assert np.array_equal(getattr(fa, f), getattr(fb, f)), f
    queries = np.concatenate([rng.standard_normal((nq // 2, dim)).astype(np.float32), rows[: nq // 2 - 1],
                              np.zeros((1, dim), np.float32)])
    assert_search_equal(ix, orc, queries, k)
    dead = rng.choice(n, n // 10, replace=False).astype(np.uint64)
    assert np.array_equal(ix.remove_ordinals(dead), orc.remove(dead))
    assert_search_equal(ix, orc, queries[:100], k)


@pytest.mark.parametrize("code,name,args", [SCALAR[0], SCALAR[3], SCALAR[4], SCALAR[6], SCALAR[8]],
                         ids=["chebyshev", "manhattan", "l3", "hamming", "minkowski3"])
@pytest.mark.parametrize("k", [3, 40])
def test_search_parity_large_leaves(code, name, args, k):
    """Leaves of up to 511 rows (the shape the fused tile kernel takes for cosine / L2): a scalar metric must route every
    visit through the gather path and still honour per-visit top-n' with ties by id."""
    z = zb()
    rng = np.random.default_rng(k + (code & 0xFF))
    n, dim = 5000, 64
    rows = clustered(rng, n, dim, centres=8)
    rows[1000:1200] = rows[:200]                 # exact duplicates: equal keys, order by id
    orc = zo.OracleIndex(dim, code, 512, 3, seed=2)
    orc.add(rows)
    ix = z.LSHIndex(dim, z.LSHIndexOptions(512, 3), metric_obj(name, args), seed=2)
    ix.add(rows)
    queries = np.concatenate([rows[:40], rng.standard_normal((24, dim)).astype(np.float32)])
    assert_search_equal(ix, orc, queries, k)                 # leaf-tile scan of the scalar metrics (seq_tile_kernel)
    st = ix.stats()
    assert st["last_tile_pairs"] == 0 and st["last_pairs"] > 0 and st["last_tiles"] > 0 and st["last_moved_bytes"] > 0
    ix.set_param("seq_tile", 0)                              # one thread per pair (score_pairs_seq_kernel): same answer
    assert_search_equal(ix, orc, queries, k)
    assert ix.stats()["last_tiles"] == 0


def test_database_facade_with_scalar_metric():
    z = zb()
    rng = np.random.default_rng(8)
    rows = clustered(rng, 800, 32)
    db = z.Database(32, z.ManhattanDistance(), index_options=z.LSHIndexOptions(5, 6), seed=3)
    docs = [i.to_bytes(8, "little") for i in range(800)]
    ids = db.insert_records(rows, docs)
    orc = zo.OracleIndex(32, zo.MANHATTAN, 5, 6, seed=3)
    orc.add(rows)
    res = db.query_vectors(rows[:30], 5)
    for q in range(30):
        eo, _ = orc.search(rows[q], 5)
        assert {int.from_bytes(d, "little") for d in res[q].values()} == set(eo.tolist())
    hit = db.index.search(rows[3], 2, z.ManhattanDistance())
    assert hit[0] == (ids[3], 0)
    with pytest.raises(ValueError):
        db.index.search(rows[3], 2, z.MinkowskiDistance(1))


def _scalar_golden():
    import glob
    import os

    here = os.path.dirname(os.path.abspath(__file__))
    return [p for p in sorted(glob.glob(os.path.join(here, "golden", "*.npz"))) if int(np.load(p)["metric"]) > zo.L2]


@pytest.mark.parametrize("path", _scalar_golden(), ids=lambda p: p.split("/")[-1])
def test_cuda_reproduces_scalar_metric_golden(path):
    """tests/golden fixtures of the scalar metrics (frozen forest, bucket keys, ids, distance bits, counts) through the
    same add / remove / add sequence over the C ABI."""
    from test_golden import cuda_reproduces_golden

    cuda_reproduces_golden(path)


def test_sharded_two_gpus_scalar_metrics_and_store_import():
    """tests/mgpu_parity_ext.py on 2 GPUs of this box: scalar metrics through the bucket-sharded store (leaf-tile scan and
    one thread per pair) and the import of an oracle-written store into a sharded index, against the unsharded oracle.
    Skipped on a single-GPU box."""
    import os
    import subprocess
    import sys

    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29519", os.path.join(root, "tests", "mgpu_parity_ext.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert out.stdout.count(": ok") == 11 and "MISMATCH" not in out.stdout
