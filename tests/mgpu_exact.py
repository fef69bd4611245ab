"""Sharded exact search: run with torchrun on G >= 2 GPUs of one node.  Every rank holds its shard (row ordinal % G == rank)
and passes the same queries; each rank's results must equal the unsharded brute force of the oracle (ordinals, distance
bits and counts bit-exact), for cosine and L2 at k = 10 and 100, after tombstones and after an incremental insert.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29513 tests/mgpu_exact.py
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
from test_gpu_exact_search import brute, clustered  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ok = True
    for mid, mname, n, dim, budget in ((zo.COSINE, "CosineDistance", 12000, 384, 0), (zo.L2, "L2Distance", 20001, 768, 2)):
        rng = np.random.default_rng(77 + n)     # same data on every rank
        rows = clustered(rng, n, dim)
        extra = clustered(rng, 1500, dim)
        queries = np.concatenate([rows[:40], clustered(rng, 60, dim)])
        ix = z.LSHIndex(dim, z.LSHIndexOptions(512, 2), getattr(z, mname)(), device=local, seed=5, shard_rank=rank,
                        shard_count=world)
        uid = [z.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ix.comm_init(uid[0])
        if budget:
            ix.set_param("exact_budget_mb", budget)   # several query chunks, each with its own allgather
        ix.add(rows)
        allrows, live = rows, np.ones(n, bool)

        def check(tag):
            nonlocal ok
            for k in (10, 100):
                _, o, b, c = ix.search_exact_batch(queries, k, want_ids=False)
                eo, eb, ec = brute(mid, allrows, live, queries, k)
                good = np.array_equal(c, ec) and np.array_equal(o, eo) and np.array_equal(b, eb)
                flags = [None] * world
                dist.all_gather_object(flags, good)
                if rank == 0:
                    print(f"[mgpu exact G={world}] {mname} n={allrows.shape[0]} dim={dim} k={k} {tag}: "
                          f"{'ok' if all(flags) else 'MISMATCH on ranks ' + str([r for r, f in enumerate(flags) if not f])}", flush=True)
                ok = ok and all(flags)

        check("bulk build")
        dead = np.arange(3, n, 10, dtype=np.uint64)
        ix.remove_ordinals(dead)
        live[dead.astype(np.int64)] = False
        check("after 10 % tombstones")
        ix.add(extra)
        allrows, live = np.concatenate([rows, extra]), np.concatenate([live, np.ones(1500, bool)])
        check("after incremental add")
        ix.close()
    dist.destroy_process_group()
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
