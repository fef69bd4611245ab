"""bench.py's command line and --dump-outputs: --steps sets the timed steps under every preset, and the dump of the last
timed step is exact, bounded and the same from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import zebra_b200 as z

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def parse(monkeypatch, *args):
    monkeypatch.setattr(sys, "argv", ["bench.py", *args])
    return bench.parse()


def test_steps_sets_the_timed_steps(monkeypatch):
    assert parse(monkeypatch).steps == 5
    assert parse(monkeypatch, "--steps", "7").steps == 7
    assert parse(monkeypatch, "--preset", "4").steps == 40            # 100M rows in 2.5M-row chunks
    assert parse(monkeypatch, "--preset", "4", "--steps", "2").steps == 2
    for bad in (["--steps", "0"], ["--warmup", "-1"], ["--dump-outputs", "d", "--workload", "hash"],
                ["--dump-outputs", "d", "--impl", "reference"]):
        with pytest.raises(SystemExit):
            parse(monkeypatch, *bad)


@pytest.mark.parametrize("mname,nq,k", [("l2", 1000, 10), ("manhattan", 300, 7), ("hamming", 50_000, 100)])
def test_dump_outputs_is_exact_masked_and_bounded(tmp_path, mname, nq, k):
    metric = bench.metric_object(z, mname)
    rng = np.random.default_rng(3)
    ords = rng.integers(0, 1 << 40, (nq, k)).astype(np.int64)
    value = 100 * rng.random((nq, k))
    bits = {64: lambda: value.view(np.uint64), 32: lambda: value.astype(np.float32).view(np.uint32).astype(np.uint64),
            0: lambda: value.astype(np.uint64)}[metric.BITS]()
    counts = rng.integers(0, k + 1, nq).astype(np.int32)
    bits[np.arange(k)[None, :] >= counts[:, None]] = np.uint64(0xFFF4000000000001)    # slots past the count: any bits
    bench.dump_outputs(str(tmp_path / "a"), metric, ords, bits.view(np.int64), counts)
    bench.dump_outputs(str(tmp_path / "b"), metric, ords, bits.view(np.int64), counts)
    names = ("ordinals", "distances", "counts", "query_rows")
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in names}
    assert sum(os.path.getsize(tmp_path / "a" / f"{n}.npy") for n in names) <= 64 << 20
    for n in names:
        assert got[n].dtype == np.float64
        assert np.array_equal(got[n], np.load(tmp_path / "b" / f"{n}.npy"), equal_nan=True)
    rows = got["query_rows"].astype(np.int64)
    assert (rows.size == nq) == (nq * 8 * (2 * k + 2) <= 64 << 20) and np.all(np.diff(rows) > 0)
    assert np.array_equal(got["counts"], counts[rows])
    live = np.arange(k)[None, :] < counts[rows][:, None]
    assert np.array_equal(got["ordinals"][live], ords[rows][live].astype(np.float64))
    assert np.all(got["ordinals"][~live] == -1) and np.all(got["distances"][~live] == np.inf)
    want = metric.to_float(bits[rows]).astype(np.float64)
    assert np.array_equal(got["distances"][live], want[live], equal_nan=True)


@pytest.mark.gpu
def test_bench_dumps_the_same_answers_twice(tmp_path):
    args = ["--gpus", "1", "--steps", "3", "--warmup", "1", "--rows", "20000", "--queries", "400", "--dim", "64",
            "--max-node-size", "256", "--trees", "2", "--cpu-seconds", "1"]
    dumps = []
    for run in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(tmp_path / run)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == 3 and line["parity_sample_ok"] and line["e2e"]["matches_device_leg"]
        dumps.append({n: np.load(tmp_path / run / f"{n}.npy") for n in ("ordinals", "distances", "counts", "query_rows")})
    assert dumps[0]["counts"].shape == (400,) and np.all(dumps[0]["counts"] > 0)
    for n in dumps[0]:
        assert np.array_equal(dumps[0][n], dumps[1][n]), n
