"""Recall of the LSH search against the exact search, and the exact search's speed, on bench.py's synthetic data.

Builds the index the way bench.py does (rows and queries from zb_synth_fill_device with the same seeds: rows seed S, queries
seed S + 1), runs the LSH search (zb_index_search_batch_device) and the exact search (zb_index_search_exact_device) on the same
queries and prints one JSON line per (forest shape, probes) (--trees and --probes take lists; probes > 0 runs the multi-probe
search, zb_index_search_probe_device):

  recall@1, recall@k         mean over all queries of recall_at_k (the exact top-k is the ground truth)
  lsh_qps, exact_qps          host clock around device-resident calls that end in a synchronise, after warm-up
  exact_pairs_per_s           live rows x queries / exact time
  exact_bytes_one_pass_per_chunk / exact_bytes_no_reuse
                              algorithmic HBM bytes: the rows once per query chunk, and once per 16-query tile (no L2 reuse)
  lsh_tile_pairs_per_s        the LSH tile kernel's own rate (last_tile_pairs / last_ms_tile_kernel), same process
  lsh_ms_plan / _scan / _total, plan_share
                              the last LSH batch's phases (zb_stats) and the plan walk's share of its total
  visits_per_query, pairs_per_query
  gpu, power_limit_w          read in the same call
  parity                      a few queries of the exact result against the oracle's brute force (bits and ordinals)

  python tools/recall_probe.py --trees 1,4,8 --probes 0,1,2,4,8 --kind 1 --queries-from held-out --out profiles/x.jsonl
Under torchrun every rank builds its shard (add_owned_device) and both searches run sharded (the exact one is collective).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import zebra_b200 as z  # noqa: E402
from oracle import zb_oracle as zo  # noqa: E402

METRICS = {"cosine": ("CosineDistance", zo.COSINE), "l2sq": ("L2SquaredDistance", zo.L2SQ), "l2": ("L2Distance", zo.L2)}


def gpu_info(local):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return out[0], float(out[1])
    except Exception:
        return torch.cuda.get_device_name(local), None


def exact_chunks(n, nq, k, dimp, filt, budget=256 << 20, sms=148, qcap=16):
    """Query chunks of one exact call (mirrors exact_plan in zb_scan.cu for the default budget, unsharded)."""
    vb = 32 + 16 * k + (32 * 8 + 5 if filt else 0)
    nr = lambda rr: -(-n // rr)  # noqa: E731
    ch = lambda rr: max(1, budget // (nr(rr) * vb + 24 + 16))  # noqa: E731
    rr = 4096
    while rr > 64 and nr(rr) * -(-min(nq, ch(rr)) // qcap) < sms * 2 * 8:
        rr //= 2
    return -(-nq // min(ch(rr), nq)), rr


def timed(fn, reps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000, help="rows over all GPUs")
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--queries", type=int, default=10_000)
    ap.add_argument("--topk", type=int, default=10)
    ap.add_argument("--metric", default="l2", choices=list(METRICS))
    ap.add_argument("--max-node-size", type=int, default=2048)
    ap.add_argument("--trees", default="4", help="comma-separated list: one index per value")
    ap.add_argument("--probes", default="0", help="comma-separated list: one LSH measurement per value and forest")
    ap.add_argument("--kind", type=int, default=1, help="synthetic rows: 0 uniform in [-1, 1), 1 clustered (bench.py's)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--queries-from", default="bench", choices=["bench", "held-out"],
                    help="bench: bench.py's queries (seed S + 1; clustered: other centres than the rows); held-out: rows n .. n + nq "
                         "of the rows' own generator (seed S), not in the index")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--parity", type=int, default=3, help="queries checked against the oracle's brute force (0: none)")
    ap.add_argument("--out", default=None, help="append the JSON lines to this file too")
    a = ap.parse_args()

    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    G, n, nq, k = world, a.rows, a.queries, a.topk
    cls, mid = METRICS[a.metric]
    name, power = gpu_info(local)
    d_q = torch.empty((nq, a.dim), dtype=torch.float32, device=dev)
    q_first, q_seed = (0, a.seed + 1) if a.queries_from == "bench" else (a.rows, a.seed)
    z.synth_fill_device(local, d_q.data_ptr(), q_first, 1, nq, a.dim, q_seed, a.kind)
    d_ord = torch.empty((nq, k), dtype=torch.int64, device=dev)
    d_bits = torch.empty((nq, k), dtype=torch.int64, device=dev)
    d_cnt = torch.empty((nq,), dtype=torch.int32, device=dev)
    for trees in (int(t) for t in a.trees.split(",")):
        ix = z.LSHIndex(a.dim, z.LSHIndexOptions(a.max_node_size, trees), getattr(z, cls)(), device=local, seed=a.seed,
                        shard_rank=rank, shard_count=G)
        if G > 1:
            uid = [z.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            ix.comm_init(uid[0])
        n_local = len(range(rank, n, G))
        d_rows = torch.empty((n_local, a.dim), dtype=torch.float32, device=dev)
        z.synth_fill_device(local, d_rows.data_ptr(), rank, G, n_local, a.dim, a.seed, a.kind)
        if G > 1:
            ix.add_owned_device(d_rows.data_ptr(), np.arange(rank, n, G, dtype=np.uint64), n)
        else:
            ix.add_device(d_rows.data_ptr(), n_local)
        del d_rows
        torch.cuda.empty_cache()

        args = (nq, d_q.data_ptr(), k, d_ord.data_ptr(), d_bits.data_ptr(), d_cnt.data_ptr())
        exact = lambda: ix.search_exact_batch_device(*args)  # noqa: E731
        for _ in range(a.warmup):
            exact()
        st_before = ix.stats()
        t_exact = timed(exact, a.reps)
        e_ord, e_bits, e_cnt = d_ord.cpu().numpy().view(np.uint64).copy(), d_bits.cpu().numpy().view(np.uint64).copy(), d_cnt.cpu().numpy().copy()
        st_after = ix.stats()
        dimp = -(-a.dim // 16) * 16
        filt = a.metric != "cosine" and k <= 16 and dimp >= 128
        chunks, range_rows = exact_chunks(n if G == 1 else -(-n // G), nq, k, dimp, filt)
        row_bytes = n * dimp * 4
        lines = []
        for probes in (int(p) for p in a.probes.split(",")):
            lsh = lambda: ix.search_batch_device(*args, probes=probes)  # noqa: E731
            for _ in range(a.warmup):
                lsh()
            t_lsh = timed(lsh, a.reps)
            st = ix.stats()
            a_ord, a_cnt = d_ord.cpu().numpy().view(np.uint64).copy(), d_cnt.cpu().numpy().copy()
            rec_k = z.recall_at_k(a_ord, a_cnt, e_ord, e_cnt)
            rec_1 = z.recall_at_k(a_ord[:, :1], np.minimum(a_cnt, 1), e_ord[:, :1], np.minimum(e_cnt, 1))
            line = {
                "rows": n, "dim": a.dim, "metric": a.metric, "kind": "clustered" if a.kind == 1 else "uniform", "queries_from": a.queries_from,
                "trees": trees, "probes": probes, "max_node_size": a.max_node_size, "queries": nq, "topk": k, "gpus": G, "gpu": name,
                "power_limit_w": power,
                "recall_at_1": float(rec_1.mean()), f"recall_at_{k}": float(rec_k.mean()), "recall_at_k_min": float(rec_k.min()),
                "lsh_s": t_lsh, "lsh_qps": nq / t_lsh, "exact_s": t_exact, "exact_qps": nq / t_exact,
                "exact_pairs_per_s": n * nq / t_exact,
                "lsh_tile_pairs_per_s": st["last_tile_pairs"] / (st["last_ms_tile_kernel"] * 1e-3) if st["last_ms_tile_kernel"] else None,
                "lsh_pairs": st["last_pairs"], "lsh_ms_tile_kernel": st["last_ms_tile_kernel"],
                "lsh_ms_plan": st["last_ms_plan"], "lsh_ms_scan": st["last_ms_scan"], "lsh_ms_total": st["last_ms_total"],
                "plan_share": st["last_ms_plan"] / st["last_ms_total"] if st["last_ms_total"] else None,
                "visits_per_query": st["last_visits"] / nq, "pairs_per_query": st["last_pairs"] / nq,
                "exact_query_chunks": chunks, "exact_range_rows": range_rows, "exact_l2_filter": filt,
                "exact_bytes_one_pass_per_chunk": row_bytes * chunks, "exact_bytes_no_reuse": row_bytes * -(-nq // 16),
                "exact_bytes_per_s_one_pass_per_chunk": row_bytes * chunks / t_exact,
                "stats_untouched_by_exact": {kk: st_before[kk] for kk in st_before if kk.startswith("last_")} ==
                                            {kk: st_after[kk] for kk in st_after if kk.startswith("last_")},
            }
            lines.append(line)
        line = lines[0]
        if a.parity and rank == 0:
            rows = zo.synth(0, 1, n, a.dim, a.seed, a.kind)
            qs = zo.synth(q_first, 1, a.parity, a.dim, q_seed, a.kind)
            ok = True
            for q in range(a.parity):
                bits = np.concatenate([zo.distance_bits_batch(mid, rows[i:i + 100_000], np.broadcast_to(qs[q], (min(100_000, n - i), a.dim)))
                                       for i in range(0, n, 100_000)])
                top = np.lexsort((np.arange(n, dtype=np.uint64), bits))[:k]
                ok &= bool(np.array_equal(e_ord[q, :e_cnt[q]], top.astype(np.uint64)) and np.array_equal(e_bits[q, :e_cnt[q]], bits[top]))
            line["parity"] = {"queries": a.parity, "bit_exact": ok}
            del rows
        if rank == 0:
            for ln in lines:
                s = json.dumps(ln)
                print(s, flush=True)
                if a.out:
                    with open(a.out, "a") as f:
                        f.write(s + "\n")
        ix.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
