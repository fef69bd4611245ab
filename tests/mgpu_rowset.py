"""Sharded restricted search: run with torchrun on G >= 2 GPUs of one node.  Every rank holds its shard (row ordinal % G ==
rank) and makes the rowset from the same list.  The whole-batch and sliced restricted LSH calls (P = 0 and P > 0) must equal
the unsharded search over the oracle (tests/probe_ref.py) with the complement of the set removed, and the restricted exact
search the brute force over the set's live rows (ordinals, distance bits and counts bit-exact), for a set below half of the
rows (compacted exact store) and one above it, after tombstones and after an incremental insert.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29515 tests/mgpu_rowset.py
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import zebra_b200 as z  # noqa: E402
from oracle import zb_oracle as zo  # noqa: E402
from probe_ref import ProbeOracle  # noqa: E402
from test_gpu_exact_search import brute, clustered  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ok = True
    for mid, mname, n, dim, mns in ((zo.COSINE, "CosineDistance", 12000, 384, 5), (zo.L2, "L2Distance", 20001, 768, 512)):
        rng = np.random.default_rng(93 + n)     # same data and sets on every rank
        rows = clustered(rng, n, dim)
        extra = clustered(rng, 1500, dim)
        queries = np.concatenate([rows[:40], clustered(rng, 61, dim)])
        twin = ProbeOracle(dim, mid, mns, 3, seed=5)
        twin.add(rows)
        ix = z.LSHIndex(dim, z.LSHIndexOptions(mns, 3), getattr(z, mname)(), device=local, seed=5, shard_rank=rank,
                        shard_count=world)
        uid = [z.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ix.comm_init(uid[0])
        ix.add(rows)
        nq = queries.shape[0]
        lo, hi = ix.slice_bounds(nq, rank, world)
        sets = []
        for frac in (0.2, 0.8):
            inset = rng.random(n) < frac
            sets.append((frac, inset, ix.rowset(ordinals=np.flatnonzero(inset))))

        def check(tag):
            nonlocal ok
            for frac, inset, rs in sets:
                allin = np.zeros(twin.rows.shape[0], bool)
                allin[:n] = inset
                ref = ProbeOracle(dim, mid, mns, 3)
                ref.load_forest(twin.rows, twin.export_forest())
                ref.remove(np.flatnonzero(~allin | twin.tomb).astype(np.uint64))
                good = True
                for k, p in ((10, 0), (10, 2), (100, 0), (33, 5)):
                    eo, eb, ec = ref.search_batch(queries, k, nthreads=8, probes=p)
                    _, o, b, c = ix.search_batch(queries, k, want_ids=False, probes=p, within=rs)
                    good = good and np.array_equal(c, ec) and np.array_equal(o, eo) and np.array_equal(b, eb)
                    _, so, sb, sc = ix.search_slice(nq, queries[lo:hi], k, want_ids=False, probes=p, within=rs)
                    good = good and np.array_equal(sc, ec[lo:hi]) and np.array_equal(so, eo[lo:hi]) and np.array_equal(sb, eb[lo:hi])
                for k in (10, 33):
                    eo, eb, ec = brute(mid, twin.rows, allin & ~twin.tomb, queries, k)
                    _, o, b, c = ix.search_exact_batch(queries, k, want_ids=False, within=rs)
                    good = good and np.array_equal(c, ec) and np.array_equal(o, eo) and np.array_equal(b, eb)
                flags = [None] * world
                dist.all_gather_object(flags, good)
                if rank == 0:
                    print(f"[mgpu rowset G={world}] {mname} dim={dim} leaves<={mns} set={frac:.0%} {tag}: "
                          f"{'ok' if all(flags) else 'MISMATCH on ranks ' + str([r for r, f in enumerate(flags) if not f])}", flush=True)
                ok = ok and all(flags)

        check("bulk build")
        dead = np.arange(3, n, 10, dtype=np.uint64)
        ix.remove_ordinals(dead)
        twin.remove(dead)
        check("after 10 % tombstones")
        ix.add(extra)
        twin.add(extra)
        check("after incremental add")
        for _, _, rs in sets:
            rs.close()
        ix.close()
    dist.destroy_process_group()
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
