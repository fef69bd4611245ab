#!/usr/bin/env python
"""bench.py -- top-k queries/sec of the LSH query hot path (BASELINE.json metric) on N B200s of one node.

A "step" is one pass of the hot path (plan -> leaf scan + top-n' -> merge) over one batch of synthetic queries
against a resident index.  N = 1 runs BASELINE config[1]: 1M x 768 f32, L2, 10k batched top-10 queries.  N > 1
is a weak-scaling run of the same per-GPU workload (1M rows and 10k queries per GPU): the forest is replicated, the
bucket-major store is sharded by bucket (leaf l lives, whole, on rank l % N), each rank plans 1/N of the queries
(NCCL allgather of the visit records), scans the visits of the leaves it owns, reduces them to a per-query local
top-k, and the local lists are merged after one NCCL allgather.

  python bench.py --gpus 1 --steps 5 --warmup 3                 # ours
  python bench.py --impl reference --gpus 1 --steps 2 --warmup 1 # the restated reference on the host cores
  python bench.py --steps 5 --warmup 3 --dump-outputs OUT       # + the last timed step's answers as OUT/*.npy

The oracle (oracle/) is used here only as the checker (sample parity) and as the measured CPU baseline.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# cosine / l2sq / l2 are the north-star metrics (fused leaf-tile scan); the rest are the scalar metrics of
# distance.rs:51-190 (gather path, one thread per pair).  Oracle ids carry the Minkowski / p-norm power in bits 8..
METRIC_IDS = {"cosine": 0, "l2sq": 1, "l2": 2, "chebyshev": 3, "canberra": 4, "bray_curtis": 5, "manhattan": 6, "l3": 7,
              "l4": 8, "hamming": 9, "minkowski3": 10 | (3 << 8), "pnorm3": 11 | (3 << 8)}
METRIC_CLASSES = {"cosine": ("CosineDistance", ()), "l2sq": ("L2SquaredDistance", ()), "l2": ("L2Distance", ()),
                  "chebyshev": ("ChebyshevDistance", ()), "canberra": ("CanberraDistance", ()),
                  "bray_curtis": ("BrayCurtisDistance", ()), "manhattan": ("ManhattanDistance", ()),
                  "l3": ("L3Distance", ()), "l4": ("L4Distance", ()), "hamming": ("HammingDistance", ()),
                  "minkowski3": ("MinkowskiDistance", (3,)), "pnorm3": ("PNormDistance", (3,))}


def metric_object(z, name):
    cls, args = METRIC_CLASSES[name]
    return getattr(z, cls)(*args)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 5; preset 4: enough to hash 100M rows)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (ordinals, distances, counts) as DIR/<name>.npy")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=1_000_000, help="rows per GPU")
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--queries", type=int, default=10_000, help="queries per GPU per step")
    ap.add_argument("--topk", type=int, default=10)
    ap.add_argument("--metric", default="l2", choices=list(METRIC_IDS))
    ap.add_argument("--max-node-size", type=int, default=2048)
    ap.add_argument("--trees", type=int, default=4)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-prefetch", action="store_true", help="end-to-end leg without zb_index_search_prefetch (uploads serialised)")
    ap.add_argument("--max-oracle-gb", type=float, default=40.0,
                    help="skip the oracle legs (parity sample, cpu_baseline) when the rows would not fit this much host memory")
    ap.add_argument("--set", action="append", default=[], help="library knob key=value (ablations)")
    ap.add_argument("--workload", default="query", choices=["query", "hash", "build"],
                    help="query = BASELINE config 2 (the default, the driver's line); hash / build = BASELINE config 4 "
                         "(bucket keys of fresh rows on a built forest / bulk insert), rows per second")
    ap.add_argument("--hash-rows", type=int, default=1_000_000, help="rows hashed per GPU per step (workload hash)")
    ap.add_argument("--flat-bits", type=int, default=0,
                    help="workload hash: K > 0 hashes FLAT tables (every level of a tree shares one plane: K bits per table, "
                         "H = K * trees planes per row, dense projection kernel) instead of the built forest")
    ap.add_argument("--delete-frac", type=float, default=0.0,
                    help="workload query: tombstone this fraction of the rows (seeded selection) before the queries, BASELINE config 5")
    ap.add_argument("--preset", type=int, default=0, choices=[0, 3, 4, 5, 6],
                    help="BASELINE.json configs at their stated sizes, as STRONG-scaling runs: 3 = 10M x 768 cosine over the GPUs, "
                         "10k top-10 queries; 4 = bucket keys of 100M x 768 rows streamed through the GPUs in 2.5M-row chunks "
                         "(workload hash; --flat-bits / --trees choose the tables); 5 = 100M x 384 L2 squared, 10 %% tombstones, "
                         "100k top-100 queries (sized for 8 GPUs); 6 = the north-star target size: 100M x 768 L2, 10k top-10 "
                         "queries (sized for 8 GPUs; 3 trees: a bucket-sharded store holds one copy of the rows per tree)")
    a = ap.parse_args()
    a.scaling = "weak"
    a.total_hash_rows = 0
    if a.preset == 4:
        a.workload, a.dim, a.rows, a.hash_rows, a.scaling = "hash", 768, 1_000_000, 2_500_000, "strong"
        a.total_hash_rows = 100_000_000
        if a.steps is None:
            a.steps = max(1, a.total_hash_rows // (a.gpus * a.hash_rows))
    elif a.preset == 6:
        a.metric, a.dim, a.topk, a.trees = "l2", 768, 10, 3
        a.rows, a.queries, a.scaling = 100_000_000 // a.gpus, max(1, 10_000 // a.gpus), "strong"
    if a.preset == 3:
        a.metric, a.dim, a.topk = "cosine", 768, 10
        a.rows, a.queries, a.scaling = 10_000_000 // a.gpus, max(1, 10_000 // a.gpus), "strong"
    elif a.preset == 5:
        a.metric, a.dim, a.topk, a.delete_frac = "l2sq", 384, 100, 0.1
        a.rows, a.queries, a.scaling = 100_000_000 // a.gpus, max(1, 100_000 // a.gpus), "strong"
    if a.steps is None:
        a.steps = 5
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and (a.impl != "ours" or a.workload != "query"):
        ap.error("--dump-outputs writes the results of the query workload of --impl ours")
    return a


def seeded_deletes(total_rows, frac, seed):
    """Ordinals to tombstone: a counter-based choice (the same list on every rank, no 100M-element permutation)."""
    out = []
    thr = int(frac * (1 << 32))
    for lo in range(0, total_rows, 1 << 24):
        o = np.arange(lo, min(total_rows, lo + (1 << 24)), dtype=np.uint64)
        h = (o + np.uint64(seed)) * np.uint64(0x9E3779B97F4A7C15)
        h ^= h >> np.uint64(29)
        h *= np.uint64(0xBF58476D1CE4E5B9)
        h ^= h >> np.uint64(32)
        out.append(o[(h & np.uint64(0xFFFFFFFF)) < np.uint64(thr)])
    return np.concatenate(out) if out else np.zeros(0, np.uint64)


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, metric, ords, bits, counts):
    """The answers of one query batch as float64 .npy files, exact (ordinals < 2^53; distances are f64 / f32 values or
    integer counts), so that two builds can be compared value for value.  Slots past a query's count hold ordinal -1 and
    distance +inf.  A batch whose answers exceed DUMP_BYTES is written for a fixed, seeded sample of its queries;
    query_rows.npy says which rows of the batch were kept."""
    nq, k = ords.shape
    rows = np.arange(nq)
    per_query = 8 * (2 * k + 2)
    if nq * per_query > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(nq, DUMP_BYTES // per_query, replace=False))
    counts = counts[rows].astype(np.int64)
    live = np.arange(k)[None, :] < counts[:, None]
    values = metric.to_float(np.where(live, bits[rows].view(np.uint64), np.uint64(0))).astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in (("ordinals", np.where(live, ords[rows].astype(np.float64), -1.0)),
                      ("distances", np.where(live, values, np.inf)),
                      ("counts", counts.astype(np.float64)), ("query_rows", rows.astype(np.float64))):
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def config_dict(a, n_gpus):
    """`config` of the JSON line: the SAME keys and values in both arms (ours and --impl reference)."""
    return {"workload": workload_name(a, n_gpus), "rows_per_gpu": a.rows, "queries_per_gpu": a.queries, "dim": a.dim,
            "top_k": a.topk, "metric": a.metric, "max_node_size": a.max_node_size, "num_trees": a.trees,
            "delete_frac": a.delete_frac, "seed": a.seed,
            "data": "synthetic: Philox clustered rows (centre[row % 4096] + 0.25 noise) and queries, seeds 0 / 1",
            "l2_policy": "every step uses a fresh query batch and streams >1 GB of rows (>> 126 MB L2)"}


def workload_name(a, n_gpus):
    return (f"{a.rows * n_gpus // 1000}k x {a.dim} f32 {a.metric.upper()} LSH index "
            f"(max_node_size {a.max_node_size}, {a.trees} trees), "
            + (f"{a.delete_frac:.0%} of the rows tombstoned, " if a.delete_frac > 0 else "")
            + f"{a.queries * n_gpus} batched top-{a.topk} queries")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (recipe of B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        if int(os.environ.get("RANK", "0")) != 0:
            return      # one poller per box: concurrent nvidia-smi loops contend for the driver and perturb the other ranks
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                                          "50", "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                                         text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2])); power.append(float(p[3]))
            except ValueError:
                continue
            for nm, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(a):
    """dram__bytes_read.sum + dram__bytes_write.sum of one tile_scan_kernel launch, from the committed ncu --set full capture
    of this same default workload (profiles/traffic.json, written by tools/profile_r1.sh); None for any other workload."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        t = json.load(open(p))
        if (t["rows"], t["dim"], t["queries"], t["metric"], t["max_node_size"], t["trees"], t["topk"]) == (
                a.rows, a.dim, a.queries, a.metric, a.max_node_size, a.trees, a.topk) and a.gpus == 1:
            return t["dram_bytes_per_launch"]
    except Exception:
        pass
    return None


# ----------------------------------------------------------------------------------------------------- reference arm
def run_reference(a):
    """The reference algorithm restated on the CPU (oracle/), all host threads, same config / metric / unit.
    Each step is a bounded sample of the step's query batch; the forest is built by the oracle itself."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import zb_oracle as zo

    cores = os.cpu_count() or 1
    n_gpus = a.gpus
    total_rows = a.rows * n_gpus
    t0 = time.time()
    rows = zo.synth(0, 1, total_rows, a.dim, a.seed, 1, cores)
    zo.set_build_threads(min(cores, a.trees))
    orc = zo.OracleIndex(a.dim, METRIC_IDS[a.metric], a.max_node_size, a.trees, seed=a.seed)
    orc.add(rows)
    if a.delete_frac > 0:
        orc.remove(seeded_deletes(total_rows, a.delete_frac, a.seed + 3))
    t_build = time.time() - t0
    nq_step = a.queries * n_gpus
    # calibrate the sample so that the whole run stays within a couple of minutes
    q0 = zo.synth(0, 1, 64, a.dim, a.seed + 1, 1, cores)
    t = time.time(); orc.search_batch(q0, a.topk, nthreads=cores); per_q = max((time.time() - t) / 64, 1e-6)
    budget = max(2.0, min(a.cpu_seconds, 90.0 / max(1, a.steps + a.warmup)))
    sample = int(max(64, min(nq_step, budget / per_q)))
    times = []
    for s in range(a.warmup + a.steps):
        q = zo.synth(s * nq_step, 1, sample, a.dim, a.seed + 1, 1, cores)
        t = time.time()
        orc.search_batch(q, a.topk, nthreads=cores)
        dt = time.time() - t
        if s >= a.warmup:
            times.append(dt)
    total = float(sum(times))
    qps = sample * len(times) / total
    line = {
        "impl": "reference", "metric": "queries_per_sec", "value": qps, "unit": "queries/s", "n_gpus": n_gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * total / len(times) * (nq_step / sample),
        "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(a, n_gpus),
        "reference_ms_per_step_is": ("measured" if sample >= nq_step else
                                     f"extrapolated from a {sample}-query sample of the {nq_step}-query step"),
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} of {nq_step} queries per step, {len(times)} steps, in-memory forest built by "
                                   f"the oracle in {t_build:.1f}s (storage engine excluded)"},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------- our arm
def gather_forest(ix, z, dist, rank, G):
    """The forest of a sharded index on rank 0: structure and planes are replicated, every rank holds the members (global
    ordinals) of its own rows; rank 0 merges the member lists leaf by leaf (ascending ordinal, D3)."""
    f = ix.export_forest()
    if G == 1:
        return f
    parts = [None] * G if rank == 0 else None
    dist.gather_object((f.leaf_off, f.members), parts, dst=0)
    if rank != 0:
        return None
    nl = f.leaf_off.size - 1
    lens = sum(np.diff(p[0]) for p in parts)
    off = np.zeros(nl + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    leaf_of = np.concatenate([np.repeat(np.arange(nl, dtype=np.int64), np.diff(p[0])) for p in parts])
    members = np.concatenate([p[1] for p in parts])
    order = np.lexsort((members, leaf_of))
    return z.Forest(f.nodes, f.roots, f.coef, f.cst, off, members[order])


def run_ours(a):
    import torch
    import torch.distributed as dist

    import zebra_b200 as z

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus and world > 1:
        raise SystemExit(f"--gpus {a.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: zebra_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    G = world
    nq = a.queries * G
    total_rows = a.rows * G
    metric = metric_object(z, a.metric)
    ix = z.LSHIndex(a.dim, z.LSHIndexOptions(a.max_node_size, a.trees), metric, device=local, seed=a.seed,
                    shard_rank=rank, shard_count=G)
    for kv in a.set:
        k, v = kv.split("=")
        ix.set_param(k, int(v))
    if G > 1:
        uid = [z.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ix.comm_init(uid[0])

    # ---- resident index: rows generated on the device, shard by shard ----
    t0 = time.time()
    n_local = len(range(rank, total_rows, G))
    d_rows = torch.empty((n_local, a.dim), dtype=torch.float32, device=dev)
    z.synth_fill_device(local, d_rows.data_ptr(), rank, G, n_local, a.dim, a.seed, 1)
    if G > 1:
        ix.add_owned_device(d_rows.data_ptr(), np.arange(rank, total_rows, G, dtype=np.uint64), total_rows)
    else:
        ix.add_device(d_rows.data_ptr(), n_local)
    del d_rows
    torch.cuda.empty_cache()
    dead = None
    if a.delete_frac > 0:   # mixed CRUD (config 5): tombstones before the queries; collective on a sharded index
        dead = seeded_deletes(total_rows, a.delete_frac, a.seed + 3)
        ix.remove_ordinals(dead)
    torch.cuda.synchronize()
    t_build = time.time() - t0

    # ---- query batches (distinct per step, so no step re-reads its predecessor's working set from L2).  A rank holds only
    #      the SLICE of every batch it fronts (queries [lo, hi) of the batch): zb_index_search_slice* ----
    nb = a.steps + a.warmup
    lo, hi = ix.slice_bounds(nq, rank, G)
    ns = hi - lo
    d_q = torch.empty((nb, ns, a.dim), dtype=torch.float32, device=dev)
    for b in range(nb):
        z.synth_fill_device(local, d_q[b].data_ptr(), b * nq + lo, 1, ns, a.dim, a.seed + 1, 1)
    h_q = d_q.cpu().pin_memory()
    d_ord = torch.empty((ns, a.topk), dtype=torch.int64, device=dev)
    d_bits = torch.empty((ns, a.topk), dtype=torch.int64, device=dev)
    d_cnt = torch.empty((ns,), dtype=torch.int32, device=dev)
    h_ord = torch.empty((ns, a.topk), dtype=torch.int64).pin_memory()
    h_bits = torch.empty((ns, a.topk), dtype=torch.int64).pin_memory()
    h_cnt = torch.empty((ns,), dtype=torch.int32).pin_memory()
    stream = torch.cuda.ExternalStream(ix.stream_ptr(), device=dev)

    def barrier():
        if G > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device(b):
        ix.search_slice_device(nq, d_q[b].data_ptr(), a.topk, d_ord.data_ptr(), d_bits.data_ptr(), d_cnt.data_ptr())

    def step_e2e(b, nxt=None):
        # double buffering through the public API: the upload of the next batch (zb_index_search_prefetch, pinned host memory)
        # overlaps this batch's scan; every batch still crosses PCIe once, inside the timed region
        if nxt is not None and not a.no_prefetch:
            ix.search_prefetch_ptr(ns, h_q[nxt].data_ptr())
        ix.search_slice_ptr(nq, h_q[b].data_ptr(), a.topk, h_ord.data_ptr(), h_bits.data_ptr(), h_cnt.data_ptr())

    # ---- device-resident leg: `value` ----
    sampler = ClockSampler(local)
    sampler.start()          # runs through warm-up, the timed region and the end-to-end leg (each only tens of ms long)
    for b in range(a.warmup):
        step_device(b)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    agg = {"scan_ms": 0.0, "plan_ms": 0.0, "select_ms": 0.0, "merge_ms": 0.0, "tile_ms": 0.0, "tiles": 0, "moved": 0, "pairs": 0, "visits": 0,
           "tile_pairs": 0, "scan_launches": 0, "launches": 0, "unique": 0, "refine_ms": 0.0, "filter_rows": 0, "filter_flagged": 0,
           "filter_used": 0, "tile_visits": 0}
    t_wall = time.perf_counter()
    e0.record(stream)
    for s in range(a.steps):
        step_device(a.warmup + s)
        st = ix.stats()
        agg["scan_ms"] += st["last_ms_scan"]; agg["plan_ms"] += st["last_ms_plan"]
        agg["select_ms"] += st["last_ms_select"]; agg["merge_ms"] += st["last_ms_merge"]
        agg["tile_ms"] += st["last_ms_tile_kernel"]; agg["tiles"] += st["last_tiles"]
        agg["moved"] += st["last_moved_bytes"]; agg["pairs"] += st["last_pairs"]; agg["visits"] += st["last_visits"]
        agg["tile_pairs"] += st["last_tile_pairs"]; agg["unique"] += st["last_unique_bytes"]
        agg["scan_launches"] += st["last_scan_launches"]; agg["launches"] += st["last_total_launches"]
        agg["refine_ms"] += st["last_ms_refine"]; agg["filter_rows"] += st["last_filter_rows"]
        agg["filter_flagged"] += st["last_filter_flagged"]; agg["filter_used"] += st["last_filter_used"]
        agg["tile_visits"] += st["last_tile_visits"]
    e1.record(stream)
    barrier()
    wall_ms = (time.perf_counter() - t_wall) * 1e3
    dev_ms = e0.elapsed_time(e1)
    t = torch.tensor([dev_ms, wall_ms], dtype=torch.float64, device=dev)
    if G > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, wall_ms = float(t[0]), float(t[1])
    ms_per_step = dev_ms / a.steps
    value = nq * a.steps / (dev_ms / 1e3)
    d_last = (d_ord.cpu(), d_bits.cpu(), d_cnt.cpu())

    # ---- end-to-end leg through the host-buffer C ABI call: H2D of the rank's query slice, D2H of its ids/distances/counts ----
    for b in range(min(3, a.warmup)):
        step_e2e(b, b + 1 if b + 1 < min(3, a.warmup) else None)
    barrier()
    t_e = time.perf_counter()
    if not a.no_prefetch:      # the first batch of the timed region is announced too (its upload has nothing to hide behind)
        ix.search_prefetch_ptr(ns, h_q[a.warmup].data_ptr())
    for s in range(a.steps):
        step_e2e(a.warmup + s, a.warmup + s + 1 if s + 1 < a.steps else None)
    barrier()
    e2e_ms = (time.perf_counter() - t_e) * 1e3
    clocks = sampler.stop()
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if G > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t[0])
    e2e_value = nq * a.steps / (e2e_ms / 1e3)
    h2d = nq * a.dim * 4                      # whole job: every query crosses PCIe once (1/G of them per rank)
    d2h = nq * a.topk * 16 + nq * 4
    same = bool(torch.equal(h_ord, d_last[0]) and torch.equal(h_bits, d_last[1]))

    # ---- roofline of the dominant kernel (the leaf scan): bytes it asks HBM for by design / its event time ----
    peak, peak_src = hbm_peak()
    # the dominant kernel = tile_scan_kernel, timed alone by CUDA events the library records around its launch on the
    # index's stream; its algorithmic bytes = sum over tiles of (leaf rows + tile queries) x 4 x dim, counted by the kernel
    scan_s = (agg["tile_ms"] if agg["tile_ms"] > 0 else agg["scan_ms"]) / 1e3
    achieved = agg["moved"] / scan_s / 1e9 if scan_s > 0 else 0.0
    traffic = ncu_traffic(a)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": "committed ncu --set full capture of this workload (profiles/traffic.json), not this run" if traffic else None,
                "peak_source": peak_src,
                "kernel": (("tile_scan3_kernel<METRIC 3> (zb_scan3_kernel.cuh: L2 through the dot-product filter; the exact second pass "
                            "refine_visits_kernel is timed separately, see l2_filter)" if agg["filter_used"] else
                            "tile_scan3_kernel (zb_scan3_kernel.cuh)") if agg["tile_ms"] > 0
                           else "score_pairs kernels (zb_kernels.cu, gather path)"),
                "algorithmic_bytes_per_launch": agg["moved"] // max(1, a.steps), "launches_per_step": 1,
                "unique_bytes_per_launch": agg["unique"] // max(1, a.steps),
                "unique_bytes_frac": (agg["unique"] / scan_s / 1e9 / peak) if scan_s > 0 else 0.0,
                "tiles_per_launch": agg["tiles"] // max(1, a.steps),
                "kernel_ms_per_launch": scan_s * 1e3 / a.steps,
                "pair_gbs": agg["pairs"] * a.dim * 4 / scan_s / 1e9 if scan_s > 0 else 0.0,
                "kernel_share_of_step": scan_s * 1e3 / dev_ms,
                "scope": "rank 0" if G > 1 else "the GPU"}

    # ---- CPU baseline (N = 1) + parity on a bounded sample of rank 0's slice of the last timed batch (every N) ----
    cpu = None
    parity = None
    host_gb = total_rows * a.dim * 4 / 1e9
    do_cpu = not a.no_cpu_baseline and host_gb <= a.max_oracle_gb   # the oracle needs every row in host memory
    forest = gather_forest(ix, z, dist, rank, G) if do_cpu else None
    if rank == 0 and do_cpu:
        from oracle import zb_oracle as zo

        cores = os.cpu_count() or 1
        rows = zo.synth(0, 1, total_rows, a.dim, a.seed, 1, cores)
        orc = zo.OracleIndex(a.dim, METRIC_IDS[a.metric], a.max_node_size, a.trees, seed=a.seed)
        orc.load_forest(rows, forest)      # same forest as the GPU arm (build parity is a separate test)
        if dead is not None:
            orc.remove(dead)
        b = a.warmup + a.steps - 1
        qh = h_q[b].numpy()
        # parity: the last timed step's batch (whose GPU results are in the host buffers) against the oracle
        tq = time.time(); orc.search_batch(qh[:64], a.topk, nthreads=cores); per_q = max((time.time() - tq) / 64, 1e-6)
        budget = 2 * a.cpu_seconds if G == 1 else 4.0
        sample = int(max(64, min(ns, budget / per_q)))   # bounded for configs far larger than the default
        tq = time.time()
        eo, eb, ec = orc.search_batch(qh[:sample], a.topk, nthreads=cores)
        dt = time.time() - tq
        go, gb, gc = h_ord.numpy()[:sample].view(np.uint64), h_bits.numpy()[:sample].view(np.uint64), h_cnt.numpy()[:sample]
        parity = bool(np.array_equal(go, eo) and np.array_equal(gb, eb) and np.array_equal(gc.astype(np.uint32), ec))
        if G == 1:
            # baseline: keep going over the other steps' batches until about cpu_seconds of CPU work is spent
            done_q, spent = sample, dt
            for bb in range(nb - 1):
                if spent >= a.cpu_seconds or sample < nq:
                    break
                tq = time.time(); orc.search_batch(h_q[bb].numpy(), a.topk, nthreads=cores); spent += time.time() - tq; done_q += nq
            cpu = {"value": done_q / spent, "unit": "queries/s", "cores": cores, "kind": "port",
                   "sample": f"{done_q} queries ({done_q // nq} of the run's {nb} batches), {spent:.1f}s on {cores} threads; "
                             "restated reference, in-memory forest (storage engine excluded)"}

    if a.dump_outputs:
        outs = [t.numpy() for t in d_last]
        if G > 1:   # every rank holds its slice of the batch; slice_bounds orders the slices by rank
            parts = [None] * G if rank == 0 else None
            dist.gather_object(outs, parts, dst=0)
            if rank == 0:
                outs = [np.concatenate([p[i] for p in parts]) for i in range(3)]
        if rank == 0:
            dump_outputs(a.dump_outputs, metric, *outs)

    per_rank = None
    if G > 1:   # per-rank phase times (ms per step): the step time is the max over ranks, these show where it goes
        mine = torch.tensor([agg[k] / a.steps for k in ("plan_ms", "scan_ms", "tile_ms", "select_ms", "merge_ms")] +
                            [agg["pairs"] / a.steps, agg["tiles"] / a.steps], dtype=torch.float64, device=dev)
        allr = [torch.zeros_like(mine) for _ in range(G)]
        dist.all_gather(allr, mine)
        per_rank = [[round(float(x), 3) for x in r] for r in allr]
    if rank == 0:
        st = ix.stats()
        line = {
            "metric": "queries_per_sec", "value": value, "unit": "queries/s", "n_gpus": G, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": a.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(a, G),
            "parallelism": (f"bucket-sharded x{G}: leaf l on rank l % {G}; every rank fronts 1/{G} of the batch (plans it, uploads / "
                            "downloads only that slice); NCCL: allgather of the query slices and of the compacted visit records, "
                            "all-to-all of per-query local top-k") if G > 1 else "single GPU",
            "index": {"build_s": round(t_build, 2), "leaves": st["leaves"], "planes": st["planes"], "device_bytes": st["device_bytes"]},
            "roofline": roofline, "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / a.steps, "matches_device_leg": same,
                    "api": ("zb_index_search_slice (host buffers)" if G > 1 else "zb_index_search_batch (host buffers)")
                           + ("" if a.no_prefetch else " + zb_index_search_prefetch of the next batch (double-buffered upload)")},
            "gpu_launches": int(agg["launches"]), "clocks": clocks,
            "phases_ms_per_step": {k: agg[k] / a.steps for k in ("plan_ms", "scan_ms", "tile_ms", "select_ms", "merge_ms")},
            "l2_filter": {"batches_filtered": agg["filter_used"], "refine_ms_per_step": agg["refine_ms"] / a.steps,
                          "exact_rows_per_visit": agg["filter_rows"] / max(1, agg["tile_visits"]),
                          "visits_rescanned_exactly_per_step": agg["filter_flagged"] / a.steps},
            "per_rank_plan_scan_tile_select_merge_ms_pairs_tiles": per_rank,
            "wall_ms_per_step": wall_ms / a.steps, "visits_per_step": agg["visits"] // a.steps,
            "pairs_per_step": agg["pairs"] // a.steps, "tile_pairs_per_step": agg["tile_pairs"] // a.steps,
            "parity_sample_ok": parity,
            "parity_sample": ("rank 0's slice of the last timed batch vs the oracle on the gathered forest" if do_cpu else
                              f"skipped: the oracle would hold {host_gb:.0f} GB of rows on the host (--max-oracle-gb {a.max_oracle_gb})"),
        }
        print(json.dumps(line), flush=True)
    if G > 1:
        dist.destroy_process_group()



# ----------------------------------------------------------------------------------------------------- config 4 workloads
def oracle_hash_parallel(orc, rows, cores):
    """oracle.hash over `cores` threads (the C call releases the GIL)."""
    from concurrent.futures import ThreadPoolExecutor

    parts = np.array_split(np.arange(rows.shape[0]), max(1, min(cores, rows.shape[0] // 64 or 1)))
    with ThreadPoolExecutor(max_workers=len(parts)) as ex:
        res = list(ex.map(lambda ix: orc.hash(rows[ix[0]:ix[-1] + 1]) if len(ix) else None, parts))
    res = [r for r in res if r is not None]
    return tuple(np.concatenate([r[i] for r in res]) for i in range(3))


def run_aux(a):
    """BASELINE config 4 (LSH projection / hashing throughput).  `hash`: bucket keys (root-to-leaf sign paths) of fresh
    rows on a built forest, rows/s.  `build`: bulk insert = level-synchronous forest build over resident rows, rows/s."""
    import torch
    import torch.distributed as dist

    import zebra_b200 as z

    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: zebra_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    G = world
    if G > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if G > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def new_index(sharded):
        ix = z.LSHIndex(a.dim, z.LSHIndexOptions(a.max_node_size, a.trees), metric_object(z, a.metric), device=local,
                        seed=a.seed, shard_rank=rank if sharded else 0, shard_count=G if sharded else 1)
        if sharded and G > 1:
            uid = [z.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            ix.comm_init(uid[0])
        for kv in a.set:
            k, v = kv.split("=")
            ix.set_param(k, int(v))
        return ix

    peak, peak_src = hbm_peak()
    nb = a.steps + a.warmup
    sampler = ClockSampler(local)
    cores = os.cpu_count() or 1
    cpu = None
    parity = None
    if a.workload == "hash":
        # forest built once from a.rows resident rows (replicated: hashing shards by row, no exchange); every step
        # hashes a fresh chunk of a.hash_rows rows per GPU that is already in HBM
        ix = new_index(False)
        d_rows = torch.empty((a.rows, a.dim), dtype=torch.float32, device=dev)
        z.synth_fill_device(local, d_rows.data_ptr(), 0, 1, a.rows, a.dim, a.seed, 1)
        flat_coef = flat_cst = None
        if a.flat_bits:
            # K-bit tables: planes through the midpoints of seeded row pairs (lsh.rs:222-225); planes are INPUT to both sides
            H = a.flat_bits * a.trees
            pick = torch.from_numpy(np.random.default_rng(a.seed + 2).integers(0, a.rows, (H, 2))).to(dev)
            pa, pb = d_rows[pick[:, 0]], d_rows[pick[:, 1]]
            coef_t = pb - pa
            flat_coef = coef_t.cpu().numpy()
            flat_cst = (-(coef_t * ((pa + pb) / 2)).sum(1)).cpu().numpy().astype(np.float32)
            ix.load_flat(d_rows.cpu().numpy(), a.flat_bits, flat_coef, flat_cst)
        else:
            ix.add_device(d_rows.data_ptr(), a.rows)
        del d_rows
        n = a.hash_rows
        # every step hashes a FRESH chunk (n rows x 4 dim bytes >> L2); the chunks live in a ring of buffers that is refilled
        # on the device between the timed sections, so 100M x 768 rows stream through one GPU without 307 GB of HBM
        ring = min(nb, max(2, int(24e9 // (n * a.dim * 4))))
        d_x = torch.empty((ring, n, a.dim), dtype=torch.float32, device=dev)

        def fill(b):
            z.synth_fill_device(local, d_x[b % ring].data_ptr(), a.rows + (b * G + rank) * n, 1, n, a.dim, a.seed, 1)

        for b in range(min(ring, nb)):
            fill(b)
        d_keys = torch.empty((n, a.trees), dtype=torch.int64, device=dev)
        d_depth = torch.empty((n, a.trees), dtype=torch.int32, device=dev)
        d_leaf = torch.empty((n, a.trees), dtype=torch.int32, device=dev)
        stream = torch.cuda.ExternalStream(ix.stream_ptr(), device=dev)
        sampler.start()
        for b in range(a.warmup):
            ix.hash_device(n, d_x[b % ring].data_ptr(), d_keys.data_ptr(), d_depth.data_ptr(), d_leaf.data_ptr())
        barrier()
        dev_ms = 0.0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s = 0
        while s < a.steps:          # timed in sections of at most `ring` steps; the refill between sections is not timed
            sec = min(ring, a.steps - s)
            for b in range(a.warmup + s, a.warmup + s + sec):
                if b >= ring:
                    fill(b)
            barrier()
            e0.record(stream)
            for b in range(a.warmup + s, a.warmup + s + sec):
                ix.hash_device(n, d_x[b % ring].data_ptr(), d_keys.data_ptr(), d_depth.data_ptr(), d_leaf.data_ptr())
            e1.record(stream)
            barrier()
            dev_ms += e0.elapsed_time(e1)
            s += sec
        h_x = d_x[(nb - 1) % ring].cpu().pin_memory()
        h_keys = np.empty((n, a.trees), dtype=np.uint64)
        barrier()
        t_e = time.perf_counter()
        e2e_steps = min(a.steps, 5)
        for s in range(e2e_steps):   # end to end: host rows in, host keys out (zb_index_hash stages through the device)
            hk, hd, hl = ix.hash(h_x.numpy())
        barrier()
        e2e_ms = (time.perf_counter() - t_e) * 1e3 * a.steps / e2e_steps
        clocks = sampler.stop()
        depth_sum = float(d_depth.sum().item())           # plane rows streamed = sum of path lengths
        units, unit_name = n * G, "rows/s"
        alg_bytes = n * (a.dim * 4 + a.trees * 16)        # each row read once + key/depth/leaf written
        extra = {"rows_per_step_per_gpu": n, "avg_depth": depth_sum / (n * a.trees),
                 "plane_bytes_from_l2_per_step": depth_sum * a.dim * 4, "fma_per_step": depth_sum * a.dim}
        kernel = "hash_kernel (zb_kernels.cu): root-to-leaf descent, one quad per (row, tree)"
        h2d, d2h = n * a.dim * 4, n * a.trees * 16
        if a.flat_bits:
            H = a.flat_bits * a.trees
            kernel = ("project3_kernel (zb_scan.cu: t3_body MODE 1, rows staged by 2-D TMA, planes resident in shared memory) + "
                      "pack_flat_keys_kernel (zb_kernels.cu, __ballot_sync)")
            extra.update({"flat_bits": a.flat_bits, "planes_per_row": H,
                          "fp32_tflops": 2.0 * a.dim * H * n * a.steps / (dev_ms / 1e3) / 1e12,
                          "fp32_peak_tflops_measured": 72.0, "fp32_peak_source": "profiles/r01_fp32_pipe.txt (FFMA, 128 lanes/clk/SM)"})
        if a.flat_bits and rank == 0 and G == 1 and not a.no_cpu_baseline:
            # the reference walks a depth-K tree per table = K point_is_above calls per (row, table): timed on one host thread
            from oracle import zb_oracle as zo

            xs = h_x.numpy()
            H = a.flat_bits * a.trees

            def cpu_keys(x):
                above = np.empty((x.shape[0], H), np.uint8)
                for h in range(H):
                    above[:, h] = zo.above_batch(np.broadcast_to(flat_coef[h], x.shape), np.full(x.shape[0], flat_cst[h], np.float32), x)
                keys = np.zeros((x.shape[0], a.trees), np.uint64)
                for t in range(a.trees):
                    for d in range(a.flat_bits):
                        keys[:, t] = (keys[:, t] << np.uint64(1)) | above[:, t * a.flat_bits + d].astype(np.uint64)
                return keys

            sample = min(n, 2048)
            t0 = time.time(); ek = cpu_keys(xs[:sample]); dt = time.time() - t0
            while dt < a.cpu_seconds / 4 and sample < n:     # grow the sample to about cpu_seconds of CPU work
                sample = min(n, sample * 4)
                t0 = time.time(); ek = cpu_keys(xs[:sample]); dt = time.time() - t0
            cpu = {"value": sample / dt, "unit": unit_name, "cores": 1, "kind": "port",
                   "sample": f"{sample} rows of the last step x {H} planes, {dt:.1f}s on 1 thread; restated point_is_above per (row, plane)"}
            parity = bool(np.array_equal(hk[:sample], ek) and np.all(hd[:sample] == a.flat_bits))
        elif rank == 0 and G == 1 and not a.no_cpu_baseline:
            from oracle import zb_oracle as zo

            orc = zo.OracleIndex(a.dim, METRIC_IDS[a.metric], a.max_node_size, a.trees, seed=a.seed)
            orc.load_forest(zo.synth(0, 1, a.rows, a.dim, a.seed, 1, cores), ix.export_forest())
            xs = h_x.numpy()
            sample = n
            t0 = time.time(); ek, ed, el = oracle_hash_parallel(orc, xs, cores); dt = time.time() - t0
            passes = 1
            while dt < a.cpu_seconds and passes < 64:   # bounded: about cpu_seconds of CPU work
                t0 = time.time(); oracle_hash_parallel(orc, xs, cores); dt += time.time() - t0; passes += 1
            cpu = {"value": sample * passes / dt, "unit": unit_name, "cores": cores, "kind": "port",
                   "sample": f"{passes} passes over the {n} rows of the last step, {dt:.1f}s on {cores} threads; restated reference descent"}
            parity = bool(np.array_equal(hk[:sample], ek) and np.array_equal(hd[:sample], ed) and np.array_equal(hl[:sample], el))
    else:
        total = a.rows * G
        n_local = len(range(rank, total, G))
        d_rows = torch.empty((n_local, a.dim), dtype=torch.float32, device=dev)
        z.synth_fill_device(local, d_rows.data_ptr(), rank, G, n_local, a.dim, a.seed, 1)
        h_rows = d_rows.cpu().pin_memory() if G == 1 else None
        ords = np.arange(rank, total, G, dtype=np.uint64)

        def build_once(host):
            """One bulk insert into a fresh index; returns (index, seconds spent in the add call alone)."""
            ix = new_index(True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if host:
                ix.add_raw(h_rows.numpy())
            elif G > 1:
                ix.add_owned_device(d_rows.data_ptr(), ords, total)
            else:
                ix.add_device(d_rows.data_ptr(), n_local)
            torch.cuda.synchronize()
            return ix, time.perf_counter() - t0

        sampler.start()
        for b in range(a.warmup):
            build_once(False)[0].close()
        barrier()
        dev_s = 0.0                   # the build is a host-driven sequence of kernels with per-level syncs: wall time of
        for s in range(a.steps):      # the insert call (index creation / destruction excluded)
            ix, dt = build_once(False)
            dev_s += dt
            if s + 1 < a.steps:
                ix.close()
            barrier()
        dev_ms = dev_s * 1e3
        e2e_ms = None
        if G == 1:
            e2e_s = 0.0
            for s in range(a.steps):
                ixh, dt = build_once(True)
                e2e_s += dt
                ixh.close()
            e2e_ms = e2e_s * 1e3
        clocks = sampler.stop()
        st = ix.stats()
        f = ix.export_forest() if G == 1 else None
        units, unit_name = total, "rows/s"
        extra = {"rows_per_gpu": a.rows, "leaves": st["leaves"], "planes": st["planes"]}
        alg_bytes = 0
        if f is not None:   # classification reads: every member of every inner node once = sum over leaves of len * depth
            depth = np.zeros(f.nodes.shape[0], dtype=np.int64)
            for i in range(f.nodes.shape[0]):
                if f.nodes[i, 0] >= 0:
                    depth[f.nodes[i, 1]] = depth[f.nodes[i, 2]] = depth[i] + 1
            leaf_nodes = np.where(f.nodes[:, 0] < 0)[0]
            lens = np.diff(f.leaf_off)[f.nodes[leaf_nodes, 3]]
            classified = int((lens * depth[leaf_nodes]).sum())
            alg_bytes = classified * a.dim * 4
            extra["classified_rows_per_build"] = classified
        kernel = "classify_kernel (zb_kernels.cu): point_is_above of every member of every node under construction"
        h2d, d2h = a.rows * a.dim * 4, 0
        if rank == 0 and G == 1 and not a.no_cpu_baseline:
            from oracle import zb_oracle as zo

            sample = min(a.rows, 2_000_000)
            rows = zo.synth(0, 1, sample, a.dim, a.seed, 1, cores)
            zo.set_build_threads(min(cores, a.trees))
            t0 = time.time()
            orc = zo.OracleIndex(a.dim, METRIC_IDS[a.metric], a.max_node_size, a.trees, seed=a.seed)
            orc.add(rows)
            dt = time.time() - t0
            cpu = {"value": sample / dt, "unit": unit_name, "cores": min(cores, a.trees), "kind": "port",
                   "sample": f"bulk build of the first {sample} rows, {dt:.1f}s, one thread per tree; restated reference, in memory"}

    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if G > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t[0])
    if rank == 0:
        sec = dev_ms / 1e3
        achieved = alg_bytes * a.steps / sec / 1e9 if alg_bytes else None
        line = {"metric": "rows_per_sec", "value": units * a.steps / sec, "unit": unit_name, "n_gpus": G, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": dev_ms / a.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"{a.workload}: {a.dim}-dim f32 rows, forest of {a.trees} trees with leaves < {a.max_node_size} "
                                       f"over {a.rows * (G if a.workload == 'build' else 1)} rows"
                                       + (f"; {units * a.steps} rows hashed in all (BASELINE config 4)" if a.workload == "hash" else ""), **extra,
                           "data": "Philox clustered, generated on device", "l2_policy": "every step streams fresh rows (>= 3 GB >> 126 MB L2)"},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak if achieved else None, "traffic": None, "peak_source": peak_src, "kernel": kernel,
                             "algorithmic_bytes_per_step": alg_bytes,
                             "fp32": ({"achieved_tflops": extra["fp32_tflops"] / G, "peak_tflops": 72.0,
                                       "frac": extra["fp32_tflops"] / G / 72.0,
                                       "binding": "fp32 FMA issue" if extra["planes_per_row"] > 20 else "hbm"}
                                      if "fp32_tflops" in extra else None),
                             "note": "whole-step time (the step is dominated by this kernel); hash: the descent also streams one "
                                     "plane row per level from L2 (plane_bytes_from_l2_per_step), which is what bounds it"},
                "cpu_baseline": cpu,
                "e2e": {"value": units * a.steps / (e2e_ms / 1e3) if e2e_ms else None, "unit": unit_name, "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": d2h},
                "gpu_launches": None, "clocks": clocks, "parity_sample_ok": parity}
        print(json.dumps(line), flush=True)
    if G > 1:
        dist.destroy_process_group()

def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.workload != "query":
        run_aux(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
