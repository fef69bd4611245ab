"""Sharded multi-probe search: run with torchrun on G >= 2 GPUs of one node.  Every rank holds its shard (row ordinal % G ==
rank).  The whole-batch call (zb_index_search_probe: every rank passes every query) and the sliced call
(zb_index_search_slice_probe: every rank passes its slice) must equal the unsharded probe rule over the oracle (tests/probe_ref.py; ordinals,
distance bits and counts bit-exact), for cosine and L2 at several (k, probes), after tombstones and after an incremental
insert.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29514 tests/mgpu_probe.py
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
from test_gpu_exact_search import clustered  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ok = True
    for mid, mname, n, dim, mns in ((zo.COSINE, "CosineDistance", 12000, 384, 5), (zo.L2, "L2Distance", 20001, 768, 512)):
        rng = np.random.default_rng(91 + n)     # same data on every rank
        rows = clustered(rng, n, dim)
        extra = clustered(rng, 1500, dim)
        queries = np.concatenate([rows[:40], clustered(rng, 61, dim)])
        orc = ProbeOracle(dim, mid, mns, 3, seed=5)
        orc.add(rows)
        ix = z.LSHIndex(dim, z.LSHIndexOptions(mns, 3), getattr(z, mname)(), device=local, seed=5, shard_rank=rank,
                        shard_count=world)
        uid = [z.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ix.comm_init(uid[0])
        ix.add(rows)
        nq = queries.shape[0]
        lo, hi = ix.slice_bounds(nq, rank, world)

        def check(tag):
            nonlocal ok
            for k, p in ((10, 1), (10, 4), (100, 2), (33, 32)):
                eo, eb, ec = orc.search_batch(queries, k, nthreads=8, probes=p)
                _, o, b, c = ix.search_batch(queries, k, want_ids=False, probes=p)
                good = np.array_equal(c, ec) and np.array_equal(o, eo) and np.array_equal(b, eb)
                _, so, sb, sc = ix.search_slice(nq, queries[lo:hi], k, want_ids=False, probes=p)
                good = good and np.array_equal(sc, ec[lo:hi]) and np.array_equal(so, eo[lo:hi]) and np.array_equal(sb, eb[lo:hi])
                flags = [None] * world
                dist.all_gather_object(flags, good)
                if rank == 0:
                    print(f"[mgpu probe G={world}] {mname} dim={dim} leaves<={mns} k={k} probes={p} {tag}: "
                          f"{'ok' if all(flags) else 'MISMATCH on ranks ' + str([r for r, f in enumerate(flags) if not f])}", flush=True)
                ok = ok and all(flags)

        check("bulk build")
        dead = np.arange(3, n, 10, dtype=np.uint64)
        ix.remove_ordinals(dead)
        orc.remove(dead)
        check("after 10 % tombstones")
        ix.add(extra)
        orc.add(extra)
        check("after incremental add")
        ix.close()
    dist.destroy_process_group()
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
