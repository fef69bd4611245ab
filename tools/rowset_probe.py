"""Restricted search (DESIGN 3.10) on bench.py's synthetic data: what a rowset costs to make and to use, and the recall of the
restricted LSH search against the restricted exact search.

Builds one unsharded index the way tools/recall_probe.py does (rows from zb_synth_fill_device, seed S; held-out queries: rows
n .. n + nq of the same generator), then for every case -- a set fraction (--fractions) and a set shape (random ordinals, one
contiguous ordinal range), plus one exclude-mode case -- prints one JSON line:

  create_s                  zb_index_rowset_from_ordinals (host list of ordinals), host clock around the call (it synchronises)
  first_call_s, derive_s    the first restricted LSH call (it derives the rowset's masks and leaf counts), and that time minus
                            the steady time of the same call: an upper bound on the derivation, since it also holds whatever
                            else differs in a first call (the unrestricted warm-up call has already sized the workspaces)
  lsh_qps_p0 / _p2          restricted LSH search (zb_index_search_rowset_device), P = 0 and 2, after warm-up
  recall_at_1 / _at_k_p*    against the restricted exact search on the same queries
  exact_qps, exact_side     restricted exact search (zb_index_search_exact_rowset_device) and which side of the half rule it
                            ran on ("compacted": the set's live rows are at most half of the slots; "masked" otherwise)
  parity                    --parity queries: the restricted LSH search (P = 0) against the oracle loaded with the same forest
                            and the complement removed, and the restricted exact search against a brute force over the set
  gpu, power_limit_w        read in the same call

  python tools/rowset_probe.py --out profiles/r05_rowset_config2.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import zebra_b200 as z  # noqa: E402
from oracle import zb_oracle as zo  # noqa: E402
from recall_probe import METRICS, gpu_info, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--queries", type=int, default=10_000)
    ap.add_argument("--topk", type=int, default=10)
    ap.add_argument("--metric", default="l2", choices=list(METRICS))
    ap.add_argument("--max-node-size", type=int, default=2048)
    ap.add_argument("--trees", type=int, default=4)
    ap.add_argument("--kind", type=int, default=1, help="synthetic rows: 0 uniform in [-1, 1), 1 clustered (bench.py's)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--fractions", default="1,0.75,0.25,0.1,0.01,0.001")
    ap.add_argument("--exclude-fraction", type=float, default=0.1, help="the exclude-mode case leaves out this fraction")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--parity", type=int, default=3, help="queries checked against the oracle (0: none)")
    ap.add_argument("--out", default=None, help="append the JSON lines to this file too")
    a = ap.parse_args()

    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    n, nq, k = a.rows, a.queries, a.topk
    cls, mid = METRICS[a.metric]
    name, power = gpu_info(0)
    d_q = torch.empty((nq, a.dim), dtype=torch.float32, device=dev)
    z.synth_fill_device(0, d_q.data_ptr(), n, 1, nq, a.dim, a.seed, a.kind)   # held-out: rows n .. n + nq of the rows' generator
    d_ord = torch.empty((nq, k), dtype=torch.int64, device=dev)
    d_bits = torch.empty((nq, k), dtype=torch.int64, device=dev)
    d_cnt = torch.empty((nq,), dtype=torch.int32, device=dev)
    ix = z.LSHIndex(a.dim, z.LSHIndexOptions(a.max_node_size, a.trees), getattr(z, cls)(), seed=a.seed)
    d_rows = torch.empty((n, a.dim), dtype=torch.float32, device=dev)
    z.synth_fill_device(0, d_rows.data_ptr(), 0, 1, n, a.dim, a.seed, a.kind)
    ix.add_device(d_rows.data_ptr(), n)
    del d_rows
    torch.cuda.empty_cache()
    args = (nq, d_q.data_ptr(), k, d_ord.data_ptr(), d_bits.data_ptr(), d_cnt.data_ptr())
    ix.search_batch_device(*args)   # the unrestricted search builds the bucket-major store before any case
    host = lambda: (d_ord.cpu().numpy().view(np.uint64).copy(), d_bits.cpu().numpy().view(np.uint64).copy(),  # noqa: E731
                    d_cnt.cpu().numpy().copy())
    rows = forest = None
    if a.parity:
        rows = zo.synth(0, 1, n, a.dim, a.seed, a.kind)
        qs = zo.synth(n, 1, a.parity, a.dim, a.seed, a.kind)
        forest = ix.export_forest()
    rng = np.random.default_rng(a.seed + 7)
    cases = []
    for f in (float(x) for x in a.fractions.split(",")):
        m = max(1, int(round(f * n)))
        cases.append(("random", f, False, np.sort(rng.choice(n, m, replace=False)) if m < n else np.arange(n)))
        lo = int(rng.integers(0, n - m + 1))
        cases.append(("range", f, False, np.arange(lo, lo + m)))
    m = int(round(a.exclude_fraction * n))
    cases.append(("exclude-random", 1 - a.exclude_fraction, True, np.sort(rng.choice(n, m, replace=False))))
    for shape, frac, excl, ords in cases:
        ords = ords.astype(np.uint64)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rs = ix.rowset(ordinals=ords, exclude=excl)
        t_create = time.perf_counter() - t0
        lsh = {p: (lambda p=p: ix.search_batch_device(*args, probes=p, within=rs)) for p in (0, 2)}
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        lsh[0]()
        torch.cuda.synchronize()
        t_first = time.perf_counter() - t0
        exact = lambda: ix.search_exact_batch_device(*args, within=rs)  # noqa: E731
        for _ in range(a.warmup):
            exact()
        t_exact = timed(exact, a.reps)
        e_ord, e_bits, e_cnt = host()
        line = {"rows": n, "dim": a.dim, "metric": a.metric, "trees": a.trees, "max_node_size": a.max_node_size, "queries": nq,
                "topk": k, "shape": shape, "fraction": frac, "exclude": excl, "count": rs.count, "gpu": name, "power_limit_w": power,
                "create_s": t_create, "first_call_s": t_first}
        for p, fn in lsh.items():
            for _ in range(a.warmup):
                fn()
            t = timed(fn, a.reps)
            a_ord, _, a_cnt = host()
            if p == 0:
                line["derive_s"] = t_first - t
            line[f"lsh_qps_p{p}"] = nq / t
            line[f"recall_at_1_p{p}"] = float(z.recall_at_k(a_ord[:, :1], np.minimum(a_cnt, 1), e_ord[:, :1], np.minimum(e_cnt, 1)).mean())
            line[f"recall_at_{k}_p{p}"] = float(z.recall_at_k(a_ord, a_cnt, e_ord, e_cnt).mean())
        line["exact_qps"] = nq / t_exact
        line["exact_side"] = "compacted" if rs.count * 2 <= n else "masked"   # unsharded, no row removed: live rows of the set = count
        if a.parity:
            inset = np.zeros(n, bool)
            inset[ords.astype(np.int64)] = True
            if excl:
                inset = ~inset
            _, lo_, lb_, lc_ = ix.search_batch(qs, k, within=rs)
            _, xo, xb, xc = ix.search_exact_batch(qs, k, within=rs)
            orc = zo.OracleIndex(a.dim, mid, a.max_node_size, a.trees, a.seed)
            orc.load_forest(rows, forest)
            dead = np.flatnonzero(~inset).astype(np.uint64)
            if dead.size:
                orc.remove(dead)
            eo, eb, ec = orc.search_batch(qs, k, nthreads=os.cpu_count() or 4)
            del orc
            ok_lsh = bool(np.array_equal(lc_, ec) and np.array_equal(lo_, eo) and np.array_equal(lb_, eb))
            ok_exact = True
            ords_in = np.flatnonzero(inset).astype(np.uint64)
            for q in range(a.parity):
                bits = zo.distance_bits_batch(mid, rows[inset], np.broadcast_to(qs[q], (ords_in.size, a.dim))) if ords_in.size else \
                    np.zeros(0, np.uint64)
                top = np.lexsort((ords_in, bits))[:k]
                ok_exact &= bool(xc[q] == top.size and np.array_equal(xo[q, :xc[q]], ords_in[top]) and np.array_equal(xb[q, :xc[q]], bits[top]))
            line["parity"] = {"queries": a.parity, "lsh_p0_bit_exact": ok_lsh, "exact_bit_exact": ok_exact}
        rs.close()
        s = json.dumps(line)
        print(s, flush=True)
        if a.out:
            with open(a.out, "a") as fh:
                fh.write(s + "\n")
    ix.close()


if __name__ == "__main__":
    main()
